"""Reference, rounding bound and float32 emulation of the bf16 tensor-core attention kernel (K5,
csrc/attention_tc.cu), shared by the GPU stage tests and the CPU test of the bound.

Per head h (32 channels), with qb = bf16(q) and R the optional key-bias table:
    s[q, k] = qb[q, h] . (k[k, h] + R[k, h]),   p = exp(s - max) over the allowed keys,   out = sum p v / sum p
The kernel's arithmetic, which `emulate` reproduces in float32: fp32 scores; per row and per 32-key quarter of each
128-key tile a running reference m (log2 units) that moves only when the tile maximum exceeds it by more than TAU = 8,
rescaling that quarter's O and l by sc = exp2(m_old - m_new); e = exp2(s log2e - m) in fp32, P = bf16(e) feeds
O += P V, l adds the fp32 e; the four quarters merge at the end and out = O (1 / l), also stored as IEEE half.

All inputs are torch tensors: q (B, Q, C), k and v (B, K, C) holding bf16 values, r (K, C) or None, allowed (B, Q, K)
bool = the effective mask (bitmap bit clear, or the row's all-masked fallback) for keys < K."""
import math

import torch

HEADS, D = 8, 32
KT = 128
TAU = 8.0
LOG2E = 1.4426950408889634
LOG2E_F32 = float(torch.tensor(LOG2E, dtype=torch.float32))     # the kernel's constant


def bf16(x):
    return x.to(torch.bfloat16).to(x.dtype)


def effective_allowed(masked, all_masked):
    """masked (B, Q, K) bool bitmap bits; all_masked (B, Q) flags or None.  A row with the flag set attends to every
    key (the reference's fallback); without flags a fully masked row attends to nothing."""
    if all_masked is None:
        return ~masked
    return ~masked | all_masked.bool()[..., None]


def _heads(x):
    return x.reshape(x.shape[:-1] + (HEADS, D)).movedim(-2, -3)        # (..., H, n, D)


def reference(q, k, v, allowed, r=None, r_abs=None, half=False, chunk=1 << 24):
    """fp64 softmax of bf16(q) (k + r) over the allowed keys, times v, and the elementwise bound of the kernel's error
        |got - ref| <= 2^-8 A + E + gamma A + 2^-22 |ref| (+ 2^-11 |ref| + 2^-25 for the half output)
    A = sum p |v| / l: P is rounded to bf16 (unit roundoff 2^-8; O uses bf16(e), l the fp32 e);
    E = sum p eps |v - ref| / l <= (sum p eps |v| + |ref| sum p eps) / l: eps bounds a score's error as a relative error
        of its p -- 2^-15 sum_d |qb| r_abs for the table (its fp32 GEMM and the hi / lo pair; r_abs = |R| +
        sum |pos + level_embed| |Wk|), 2^-19 sum_d |qb| |k| for the fp32 accumulation, 2^-22 (|s| + |max|) for
        s log2e - m in fp32, 2^-19 for ex2.approx and the merge factors;
    gamma = (K/4 + 64 + ntiles) 2^-24: O's fp32 accumulation and its rescale multiplications.
    Returns ref, bound, both (B, Q, C) float64, and p_max (B, Q, H), the largest weight of each row (1 = one-hot).
    A row without an allowed key has ref = 0 and bound = 0."""
    B, Q, C = q.shape
    K = k.shape[1]
    qb = _heads(bf16(q.float()).double())                                 # (B, H, Q, D)
    kd, vd = _heads(k.double()), _heads(v.double())                       # (B, H, K, D)
    kr = kd + _heads(r.double())[None] if r is not None else kd
    ra = _heads(r_abs.double())[None] if r_abs is not None else None
    ntiles = (K + KT - 1) // KT
    gamma = (K / 4 + 64 + ntiles) * 2.0 ** -24
    ref = torch.zeros((B, HEADS, Q, D), dtype=torch.float64)
    bnd = torch.zeros_like(ref)
    pmax = torch.zeros((B, HEADS, Q), dtype=torch.float64)
    step = max(1, chunk // max(1, K * HEADS * B))
    for q0 in range(0, Q, step):
        sl = slice(q0, min(Q, q0 + step))
        qs = qb[:, :, sl]
        al = allowed[:, None, sl].expand(B, HEADS, -1, K)
        s = qs @ kr.transpose(-1, -2)
        sm = s.masked_fill(~al, -math.inf)
        m = sm.amax(-1, keepdim=True)
        live = torch.isfinite(m)
        p = torch.where(al, torch.exp(sm - torch.where(live, m, torch.zeros_like(m))), torch.zeros_like(s))
        l = p.sum(-1, keepdim=True)
        linv = torch.where(l > 0, 1.0 / l.clamp(min=1e-300), torch.zeros_like(l))
        o = (p @ vd) * linv
        a = (p @ vd.abs()) * linv
        eps = 2.0 ** -19 * (qs.abs() @ kd.abs().transpose(-1, -2)) + 2.0 ** -22 * (s.abs() + m.abs().nan_to_num(0, 0, 0)) \
            + 2.0 ** -19
        if ra is not None:
            eps = eps + 2.0 ** -15 * (qs.abs() @ ra.transpose(-1, -2))
        pe = p * eps
        e = ((pe @ vd.abs()) + o.abs() * pe.sum(-1, keepdim=True)) * linv
        b = 2.0 ** -8 * a + e + gamma * a + 2.0 ** -22 * o.abs()
        if half:
            b = b + 2.0 ** -11 * o.abs() + 2.0 ** -25
        ref[:, :, sl], bnd[:, :, sl] = o, torch.where(l > 0, b, torch.zeros_like(b))
        pmax[:, :, sl] = (p.amax(-1) * linv[..., 0])
    back = lambda x: x.movedim(-3, -2).reshape(B, Q, C)
    return back(ref), back(bnd), pmax.movedim(1, 2)


def emulate(q, k, v, allowed, r_hi=None, r_lo=None, mutant=None):
    """float32 emulation of the kernel's arithmetic (see the module docstring).  Keys past K up to the tile boundary
    are masked by the kernel's tail mask; mutant='tail' unmasks them (their K, V and R rows are TMA zero fill).
    Other mutants: 'p_trunc' (P truncated to bf16), 'sc_one' (no rescale).  Returns (out fp32, out half)."""
    B, Q, C = q.shape
    K = k.shape[1]
    ntiles = (K + KT - 1) // KT
    Kp = ntiles * KT
    pad = lambda x: torch.cat([x, torch.zeros(x.shape[:-2] + (Kp - K, x.shape[-1]), dtype=x.dtype)], -2)
    qb = _heads(bf16(q.float()).double())
    kr = _heads(pad(k.double()))
    if r_hi is not None:
        kr = kr + _heads(pad(r_hi.double()))[None]
        if r_lo is not None:
            kr = kr + _heads(pad(r_lo.double()))[None]
    vf = _heads(pad(v.float()))                                           # (B, H, Kp, D)
    s = (qb @ kr.transpose(-1, -2)).float()                               # (B, H, Q, Kp): fp32 scores
    al = torch.zeros((B, Q, Kp), dtype=torch.bool)
    al[:, :, :K] = allowed
    if mutant == 'tail':
        al[:, :, K:] = True
    s = s.masked_fill(~al[:, None], -math.inf)
    log2e = torch.tensor(LOG2E, dtype=torch.float32)
    parts = []
    for cq in range(4):
        m_ref = torch.full((B, HEADS, Q), -math.inf, dtype=torch.float32)
        l = torch.zeros((B, HEADS, Q), dtype=torch.float32)
        o = torch.zeros((B, HEADS, Q, D), dtype=torch.float32)
        for t in range(ntiles):
            k0 = t * KT + cq * 32
            st = s[..., k0:k0 + 32]
            mx = st.amax(-1) * log2e
            move = mx > m_ref + TAU
            fix = move & (m_ref != -math.inf)
            if mutant != 'sc_one':
                sc = torch.where(fix, torch.exp2(m_ref - mx), torch.ones_like(mx))
                o = o * sc[..., None]
                l = l * sc
            m_ref = torch.where(move, mx, m_ref)
            mneg = torch.where(m_ref == -math.inf, torch.zeros_like(m_ref), -m_ref)
            e = torch.exp2((st.double() * LOG2E_F32 + mneg[..., None].double()).float())     # one fma rounding
            if mutant == 'p_trunc':
                pb = (e.view(torch.int32) & ~0xFFFF).view(torch.float32)
            else:
                pb = bf16(e)
            o = o + pb @ vf[:, :, k0:k0 + 32]
            l = l + e.sum(-1)
        parts.append((m_ref, l, o))
    m = parts[0][0]
    for p in parts[1:]:
        m = torch.maximum(m, p[0])
    l_tot = torch.zeros_like(m)
    o_tot = torch.zeros_like(parts[0][2])
    for m1, l1, o1 in parts:
        a1 = torch.where(m1 == -math.inf, torch.zeros_like(m1), torch.exp2(m1 - m))
        l_tot = l_tot + l1 * a1
        o_tot = o_tot + o1 * a1[..., None]
    inv = torch.where(l_tot > 0, 1.0 / l_tot, torch.zeros_like(l_tot))
    out = (o_tot * inv[..., None]).movedim(1, 2).reshape(B, Q, C)
    return out, out.half()


def key_bias_table(sd, layer, h, w, num_levels=3):
    """fp64 key-bias table of decoder layer `layer` on a (h, w) level: R = (pos + level_embed) Wk^T + bk, and
    r_abs = |R| + |pos + level_embed| |Wk|^T for the bound.  sd: a reference-keyed state dict."""
    from oracle.cgg_oracle import sine_pos_enc
    C = sd['level_embed.weight'].shape[1]
    p = 'transformer_decoder.layers.%d.attentions.0.attn.' % layer
    wk = sd[p + 'in_proj_weight'][C:2 * C].double()
    bk = sd[p + 'in_proj_bias'][C:2 * C].double()
    x = sine_pos_enc(h, w, C // 2).double() + sd['level_embed.weight'][layer % num_levels].double()
    r = x @ wk.t() + bk
    return r, r.abs() + x.abs() @ wk.abs().t()


def split_hi_lo(r):
    """The table as the kernel holds it: fp32 values as a bf16 (hi, lo) pair."""
    r32 = r.float()
    hi = r32.bfloat16().float()
    return hi.double(), (r32 - hi).bfloat16().double()


# ---------------------------------------------------------------------------------------------- shared cases
def random_mask(g, B, Q, K, density, blob=False, keep=()):
    """(B, Q, K) bitmap bits: random at `density`, or (blob) one window of allowed keys per row, so that most 128-key
    tiles are masked for every query; the keys in `keep` are allowed everywhere.  Then row (0, 0) is wholly masked (a
    fallback row) and row (B-1, 5) masks the first half of the keys."""
    if blob:
        masked = torch.ones((B, Q, K), dtype=torch.bool)
        start = torch.randint(0, max(1, K // 8), (B, Q), generator=g)
        width = max(1, int(K * (1 - density) / 4))
        idx = torch.arange(K)
        masked &= ~((idx >= start[..., None]) & (idx < start[..., None] + width))
    else:
        masked = torch.rand((B, Q, K), generator=g) < density
    masked[:, :, list(keep)] = False
    masked[0, 0] = True
    masked[B - 1, min(5, Q - 1), :K // 2] = True
    return masked


def ramp_case(g, B, Q, K, log2_per_tile):
    """Scores that climb (or fall) through one channel of K: q's last channel of every head is 1, K's is
    bf16(ramp * key), so each 128-key tile moves the row maximum by about log2_per_tile (log2 units).  Up by 10: every
    tile moves the lazy reference, with 0 < sc ~ 2^-10; down: no move after the first tile; up by 7.5: P grows up to
    2^7.5 before the reference moves."""
    C = HEADS * D
    q = torch.randn((B, Q, C), generator=g) * 0.25
    k = torch.randn((B, K, C), generator=g)
    v = torch.randn((B, K, C), generator=g)
    ramp = torch.arange(K, dtype=torch.float64) * (log2_per_tile / LOG2E / KT)
    if log2_per_tile < 0:
        ramp = ramp - ramp[-1]
    for h in range(HEADS):
        q[..., h * D + D - 1] = 1.0
        k[..., h * D + D - 1] = ramp.float()
    return q, bf16(k), bf16(v)


TWO_LEVEL_ANCHORS = (0, 32, 64, 96)


def two_level_case(g, B, Q, K):
    """Exact scores: q is the unit vector of each head's channel 0, and K's channel 0 is 0 at the anchor keys 0, 32,
    64, 96 (the first key of each quarter of the first tile; allowed in every row, see random_mask's keep) and -0.6875
    elsewhere.  Every quarter's reference is then 0 from the first tile on, each other key has e = exp(-0.6875) =
    0.50283, which is 0.50390625 in bf16 rounded to nearest (2^-8.9 relative) and 0.5 truncated (2^-7.5), far from a
    rounding midpoint, and V is a positive integer, so the bound's 2^-8 term of P's rounding is what a truncated P
    exceeds."""
    C = HEADS * D
    q = torch.zeros((B, Q, C))
    k = torch.randn((B, K, C), generator=g)
    for h in range(HEADS):
        q[..., h * D] = 1.0
        k[..., h * D] = -0.6875
        k[:, [a for a in TWO_LEVEL_ANCHORS if a < K], h * D] = 0.0
    v = torch.randint(1, 9, (B, K, C), generator=g).float()
    return q, bf16(k), v
