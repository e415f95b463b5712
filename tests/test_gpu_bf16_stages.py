"""Stage tests of the bf16 (tcgen05) head call: each GEMM stage against a reference of its OWN arithmetic, in fp64 on
the CPU, at the shapes where the kernels change route.  The end-to-end tests of test_gpu_bf16.py hold the product to
BASELINE's statistical bars (1e-2 of range, 99.9 % of the attention-mask bits); here the bars come from the rounding
steps of each stage, so a dropped term, a wrong row offset or a wrong rounding mode fails although the product bars
would still pass.

  K1  query heads        post_norm -> [v2l | mask_embed.0 | cls] -> mask_embed.2 -> .4, hi/lo bf16 operand pairs
  K2  mask einsum        mask[call, b, q, p] = sum_c bf16(me)[b, call, q, c] mf[b, c, p]            (bf16 output)
  K3  attention-mask     bit = sum_c fp16(me)[b, q, c] fds_l[b, c, key] <= MASKED_LOGIT_MAX            (fp32 accumulate)
  K4  K/V projection     kv_l[b, key, :] = mem_l[b, :, key] [Wk; Wv]^T (+ level_embed Wv^T + bv on V)   (bf16 output)

Workspace layouts the tests read (each test asserts the one it relies on, so that a layout change fails loudly):
  me_all  (TcWs::carve, store_me_kernel): rows [image][call * q_pad + q], 2C wide; columns [0, C) bf16(me) (K2),
          [C, 2C) fp16(me) (K3); rows_per_batch = (L + 1) * q_pad
  fds_l   (B, C, pitch8(K_l)) fp16, the level-l resample of the mask features
  kv_l    (B, K_l, nl * 2C) bf16: layer slot sl's K in columns [sl C, (sl+1) C), its V in [(nl+sl) C, (nl+sl+1) C)
"""
import numpy as np
import pytest
import torch

from cgg_b200 import synth
from cgg_b200.head import build_head_from_state_dict

pytestmark = pytest.mark.gpu
DEV = 'cuda'
C = 256
L = 9
CALLS = L + 1
NL = 3                                                 # layers reading each level (9 layers over 3 levels)
RATIOS = (8, 4, 2)                                     # mask-feature pixels per key side at levels 0, 1, 2
MASKED_LOGIT_MAX = float(np.float32(-1.7881392e-07))  # common.cuh: sigmoid(x) < 0.5 in fp32 <=> x <= this
NAN16 = 0x7FC0                                         # a NaN as bf16 and as fp16


def q_pad(Q):
    """B-operand rows per head call: the mask-einsum routing table of tc_create (gemm_tc.cu)."""
    r8, r16 = (Q + 7) // 8 * 8, (Q + 15) // 16 * 16
    if Q <= 104:                  # tc_einsum_t_kernel, two head calls per step
        return max(16, r8)
    if Q <= 208:                  # 105..128: pair kernel, one N tile; 129..208: tc_einsum_t_kernel split over the pair
        return r16
    T = (Q + 207) // 208          # pair kernel, T N tiles of round16(ceil(Q / T)) per head call
    return T * (((Q + T - 1) // T + 15) // 16 * 16)


def level_resample_ref(mf, ratio):
    """The bf16 path's resample of the mask features to a level (downsample3_kernel): F.interpolate(bilinear,
    align_corners=False) at an exact integer ratio reads the central 2x2 of each ratio x ratio block with weights 1/2,
    evaluated as 0.5 (0.5 a + 0.5 b) + 0.5 (0.5 c + 0.5 d) in fp32.  mf (B, C, H4, W4) -> (B, C, H4/r, W4/r) fp32."""
    B, Cc, H4, W4 = mf.shape
    x = mf.float().view(B, Cc, H4 // ratio, ratio, W4 // ratio, ratio)
    o = ratio // 2 - 1
    a, b = x[:, :, :, o, :, o], x[:, :, :, o, :, o + 1]
    c, d = x[:, :, :, o + 1, :, o], x[:, :, :, o + 1, :, o + 1]
    return 0.5 * (0.5 * a + 0.5 * b) + 0.5 * (0.5 * c + 0.5 * d)


def _unpack(bm, nbits):
    """(B, Q, W32) int32 bitmap -> (B, Q, nbits) bool, key k = bit k % 32 of word k // 32."""
    w = bm.cpu().numpy().astype(np.int32)
    bits = np.unpackbits(w.view(np.uint8), bitorder='little').reshape(w.shape[0], w.shape[1], -1)[:, :, :nbits]
    return torch.from_numpy(bits.astype(bool))


def _head(Q, seed=3, ncls1=49, sd=None):
    sd = sd if sd is not None else synth.make_params(seed=seed, num_queries=Q, perturb=True, num_classes_p1=ncls1)
    return build_head_from_state_dict(sd, Q, ncls1, 'bf16', DEV)


class _Stage:
    """A bf16 head's runtime prepared for one input size and batch, with views of its workspace buffers."""

    def __init__(self, head, H, W, B):
        self.rt = head._runtime(torch.device(DEV, 0))
        self.Q, self.B = head.num_queries, B
        (self.H4, self.W4), self.sizes = synth.level_sizes(H, W)
        self.K = [h * w for h, w in self.sizes]
        self.rt.prepare(self.H4, self.W4, self.sizes, B)
        self.q_pad = q_pad(self.Q)
        self.rows_per_batch = CALLS * self.q_pad

    def _buf(self, name, nbytes):
        off = self.rt.lib.cgg_workspace_offset(self.rt.handle, self.B, name.encode())
        assert off + nbytes <= self.rt.workspace.numel(), name
        return self.rt.workspace[off:off + nbytes]

    def me_all(self):
        """(B, rows_per_batch, 2C) int16 view of the all-call mask-embedding operand."""
        n = self.B * self.rows_per_batch * 2 * C
        return self._buf('me_all', 2 * n).view(torch.int16).view(self.B, self.rows_per_batch, 2 * C)

    def fds(self, level):
        p = (self.K[level] + 7) // 8 * 8
        return self._buf('fds%d' % level, self.B * C * p * 2).view(torch.float16).view(self.B, C, p)

    def kv(self, level):
        n = self.B * self.K[level] * NL * 2 * C
        return self._buf('kv%d' % level, 2 * n).view(torch.bfloat16).view(self.B, self.K[level], NL * 2 * C)

    def assert_me_all_layout(self, me):
        """head_call writes call slot 0: rows [0, Q) of images 0 and 1 hold bf16(me) | fp16(me) of its returned me."""
        rows = self.me_all().cpu()
        for b in (0, 1):
            assert torch.equal(rows[b, :self.Q, :C], me[b].cpu().bfloat16().view(torch.int16)), ('bf16(me) rows', b)
            assert torch.equal(rows[b, :self.Q, C:], me[b].cpu().half().view(torch.int16)), ('fp16(me) rows', b)

    def assert_fds_exact(self, mf):
        """fds_l[:, :, :K_l] == fp16(level_resample_ref) bit for bit (the padding columns are not compared)."""
        for level, r in enumerate(RATIOS):
            want = level_resample_ref(mf, r).half().reshape(self.B, C, -1)
            got = self.fds(level)[:, :, :self.K[level]].cpu()
            bad = int((got.view(torch.int16) != want.view(torch.int16)).sum())
            assert bad == 0, 'level %d: %d resampled features differ' % (level, bad)


def _bf16_randn(g, shape):
    return torch.randn(shape, generator=g).bfloat16()


# ---------------------------------------------------------------------------------------------------- K2, exact
K2_QS = [8, 37, 104, 105, 128, 129, 200, 208, 209, 256, 300, 512]
CALL_RANGES = [(0, 10), (1, 3), (9, 1), (2, 5)]
SENTINEL = 0.1                                         # not an integer: an einsum output never equals it


@pytest.mark.parametrize('Q', K2_QS)
def test_k2_mask_einsum_exact_on_integer_operands(Q):
    """K2 with me and the mask features in {-1, 0, 1}: every sum is an integer of magnitude <= 256, exact in bf16 and in
    the fp32 accumulator, so the output must EQUAL the reference.  Every operand row the call must not read -- pad rows
    q >= Q of each call slot, call slots outside the range, the fp16 half -- holds NaN, so a wrong call, image or row
    offset shows as NaN or as a wrong integer; a plane past the range keeps its sentinel.  The query counts reach every
    route of the table in q_pad() and both sides of each boundary; 352x288 has a partial last pixel tile / pair."""
    head = _head(Q)
    g = torch.Generator().manual_seed(Q)
    for H, W in ((256, 256), (352, 288)):
        for B in (1, 3):
            st = _Stage(head, H, W, B)
            HW = st.H4 * st.W4
            mf = torch.randint(-1, 2, (B, C, st.H4, st.W4), generator=g).bfloat16()
            mfd = mf.to(DEV)
            if B == 3:
                _, _, _, me, _, _ = st.rt.head_call(torch.randn((B, Q, C), generator=g).to(DEV), mfd, 0, want_bits=False)
                st.assert_me_all_layout(me)
            me = torch.randint(-1, 2, (B, CALLS, Q, C), generator=g).float()
            # fp32 products of small integers are exact in any summation order: this IS the fp64 einsum
            ref = torch.matmul(me.view(B, CALLS * Q, C), mf.float().view(B, C, HW)).view(B, CALLS, Q, HW)
            ref = ref.transpose(0, 1).bfloat16().float()                           # (calls, B, Q, HW)
            assert float(ref.abs().max()) <= 256
            me_bits = me.bfloat16().view(torch.int16)
            for first, n in CALL_RANGES:
                rows = torch.full((B, CALLS, st.q_pad, 2 * C), NAN16, dtype=torch.int16)
                rows[:, first:first + n, :Q, :C] = me_bits[:, first:first + n]
                st.me_all().copy_(rows.view(B, st.rows_per_batch, 2 * C))
                outs = []
                for _ in range(2):
                    out = torch.full((n + 1, B, Q, st.H4, st.W4), SENTINEL, dtype=torch.bfloat16, device=DEV)
                    st.rt.mask_einsum(mfd, out, first_call=first, num_calls=n)
                    outs.append(out.cpu())
                assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16)), ('run to run', H, W, B, first, n)
                got = outs[0]
                assert bool((got[n] == SENTINEL).all()), ('plane past the range written', H, W, B, first, n)
                for i in range(n):
                    gi = got[i].float().view(B, Q, HW)
                    if not torch.equal(gi, ref[first + i]):
                        bad = (gi != ref[first + i])
                        raise AssertionError('Q=%d %dx%d B=%d calls (%d, %d): plane %d, %d of %d outputs differ (%d NaN)'
                                             % (Q, H, W, B, first, n, i, int(bad.sum()), bad.numel(),
                                                int(gi.isnan().sum())))


# ------------------------------------------------------------------------------------------- K2, production feed
@pytest.mark.parametrize('Q', [100, 128, 200, 300])
def test_k2_production_feed_within_rounding_bound(Q):
    """The ten masks of a free-running bf16 forward against einsum(bf16(me_j), mf) in fp64, me_j recomputed by
    head_call from the forward's decoder state (bitwise the forward's own, test_gpu_bf16._batched_einsum_check).
    Bound: |got - ref| <= 2^-8 |ref| + 2^-14 sum_c |bf16(me)| |mf|, i.e. the round-to-nearest of the output to bf16
    (8-bit significand: relative error up to 2^-8, reached by a correct kernel -- 0.9 x 2^-8 measured) plus the fp32
    accumulation of 256 exact products (<= 256 * 2^-24 = 2^-16 of the absolute sum; 4x margin).  This pins
    store_me_kernel's round-to-nearest (truncating me to bf16 gives ~16x the bound) and the call-slot placement."""
    B, H, W = 2, 256, 256
    head = _head(Q, seed=13)
    mf, mems = synth.make_inputs(4, B, H, W, dtype=torch.bfloat16)
    mfd, memd = mf.to(DEV), [m.to(DEV) for m in mems]
    _, _, mask, dbg = head.decoder_forward(mfd, memd, return_debug=True)
    st = _Stage(head, H, W, B)
    HW = st.H4 * st.W4
    f = mf.double().view(B, C, HW)
    for j in range(CALLS):
        _, _, _, me, _, _ = st.rt.head_call(dbg['x'][j].contiguous(), mfd, j % 3, want_bits=False)
        if j == 0:
            st.assert_me_all_layout(me)
        e = me.cpu().bfloat16().double()
        ref = torch.matmul(e, f)
        bound = 2.0 ** -8 * ref.abs() + 2.0 ** -14 * torch.matmul(e.abs(), f.abs())
        err = (mask[j].cpu().double().view(B, Q, HW) - ref).abs()
        worst = float((err / bound).max())
        assert worst <= 1.0, 'head call %d: error %.3g of the bound' % (j, worst)


# ------------------------------------------------------------------------------------------ level resample, exact
@pytest.mark.parametrize('H,W', [(256, 256), (352, 288), (1056, 800)])
def test_level_resample_exact(H, W):
    """fds0..2 after a head call equal fp16(level_resample_ref) bit for bit.  1056x800 has key counts 825 / 3300 /
    13200: the first two planes are padded to a pitch of 8."""
    B, Q = 2, 100
    head = _head(Q)
    st = _Stage(head, H, W, B)
    g = torch.Generator().manual_seed(H + W)
    mf = _bf16_randn(g, (B, C, st.H4, st.W4))
    for level in range(3):
        st.fds(level).view(torch.int16).fill_(NAN16)
    st.rt.head_call(torch.randn((B, Q, C), generator=g).to(DEV), mf.to(DEV), 0)
    st.assert_fds_exact(mf)


# ------------------------------------------------------------------------------------------------- K3 bits
BITS_QS = [8, 37, 100, 128, 200, 256, 257, 300, 512]
FP16_MIN_NORMAL = 2.0 ** -14


def _check_bits(st, level, bm, am):
    """The returned bitmap as (B, Q, K) bool; the bits past the last key of the last word must be clear, and
    all_masked must be "the row's popcount == K" of the bitmap."""
    K = st.K[level]
    allbits = _unpack(bm, (K + 31) // 32 * 32)
    assert not allbits[:, :, K:].any(), 'bits past the last key'
    bits = allbits[:, :, :K]
    assert torch.equal(am.cpu().bool(), bits.sum(-1) == K), 'all_masked != (popcount == K)'
    return bits


def _plant(mf, me16, level, K, wl):
    """Planted keys, whose logits are exact: every 8th key has zero features in every channel (logit 0: unmasked), and
    half the keys are nonzero in one channel c only, with a power of two s in the fp16 normal range.  Each such pair of
    keys comes from a query q with a small fp16 normal me[q, c] and takes s = -sign(me) 2^e, 2^(e+1) with
    |me| 2^e <= |MASKED_LOGIT_MAX| < |me| 2^(e+1): a negative logit just above the cut-off and one below it.
    Returns the new mask features and, per image, (keys, channels, values) of the single-channel keys."""
    B = mf.shape[0]
    r = RATIOS[level]
    h = mf.shape[2] // r
    kval = torch.zeros((B, C, K))
    planted = torch.zeros((B, K), dtype=torch.bool)
    singles = []
    keys = torch.arange(K)
    planted[:, keys % 8 == 0] = True
    ks = keys[(keys % 8 >= 1) & (keys % 8 <= 4)]
    for b in range(B):
        a = me16[b].abs()
        cand = ((a >= FP16_MIN_NORMAL) & (a * FP16_MIN_NORMAL <= -MASKED_LOGIT_MAX)).nonzero()
        assert len(cand) > 0, 'no small fp16-normal mask embedding to plant against'
        chans, vals = [], []
        for i, k in enumerate(ks.tolist()):
            q, c = cand[(i // 2) % len(cand)].tolist()
            m = float(me16[b, q, c])
            e = int(np.floor(np.log2(-MASKED_LOGIT_MAX / abs(m)))) + i % 2
            s = -np.sign(m) * 2.0 ** e
            assert FP16_MIN_NORMAL <= abs(s) <= 1.0
            kval[b, c, k] = s
            chans.append(c)
            vals.append(s)
        planted[b, ks] = True
        singles.append((ks, torch.tensor(chans), torch.tensor(vals, dtype=torch.float64)))
    up = lambda t: t.view(t.shape[0], t.shape[1], h, -1).repeat_interleave(r, 2).repeat_interleave(r, 3)
    mfp = torch.where(up(planted[:, None]), up(kval), mf.float()).bfloat16()
    return mfp, singles


@pytest.mark.parametrize('Q', BITS_QS)
def test_k3_attention_mask_bits(Q):
    """K3 (tc_bits_kernel: one query slice up to 256 queries, two above) against the fp64 logit
    sum_c fp16(me)[q, c] fds[c, key], with head_call's me and the fds checked bit for bit against the resample reference.
      random inputs: a bit may disagree with (logit <= MASKED_LOGIT_MAX) only inside the band
        |logit - MASKED_LOGIT_MAX| <= 2^-14 sum_c |fp16(me)| |fds| (fp32 accumulation of exact fp16 x fp16 products:
        <= 256 * 2^-24 = 2^-16 of the absolute sum, 4x margin); all_masked matches the reference on rows without band
        entries;
      planted keys (_plant): logits are exact, so the bits must equal the reference (pairs whose fp16(me) is subnormal
        are skipped: whether the tensor core keeps fp16 subnormals is not asked here);
      a constant image: every key of a row has the same logit, so each row is wholly masked or wholly unmasked, and
        all_masked matches the reference outside the band."""
    head = _head(Q, seed=5)
    g = torch.Generator().manual_seed(100 + Q)
    for H, W in ((256, 256), (352, 288)):
        for B in (1, 3):
            st = _Stage(head, H, W, B)
            x = torch.randn((B, Q, C), generator=g).to(DEV)
            mf = _bf16_randn(g, (B, C, st.H4, st.W4))
            n_above = n_below = 0
            for level in range(3):
                K, wl = st.K[level], st.sizes[level][1]
                what = 'Q=%d %dx%d B=%d level %d' % (Q, H, W, B, level)
                # ---- random inputs
                _, _, _, me, bm, am = st.rt.head_call(x, mf.to(DEV), level)
                if level == 0:
                    st.assert_fds_exact(mf)
                e = me.cpu().half().double()
                f = st.fds(level)[:, :, :K].cpu().double()
                logit = torch.matmul(e, f)
                band = 2.0 ** -14 * torch.matmul(e.abs(), f.abs())
                want = logit <= MASKED_LOGIT_MAX
                inband = (logit - MASKED_LOGIT_MAX).abs() <= band
                bits = _check_bits(st, level, bm, am)
                bad = (bits != want) & ~inband
                assert not bad.any(), '%s: %d bits outside the band disagree' % (what, int(bad.sum()))
                clear = ~inband.any(-1)
                assert torch.equal(am.cpu().bool()[clear], want.all(-1)[clear]), what + ': all_masked'
                # ---- planted keys with exact logits
                mfp, singles = _plant(mf, e, level, K, wl)
                _, _, _, me2, bm, am = st.rt.head_call(x, mfp.to(DEV), level)
                assert torch.equal(me2, me), what + ': me changed with the mask features'
                bits = _check_bits(st, level, bm, am)
                assert not bits[:, :, torch.arange(K) % 8 == 0].any(), what + ': a zero-feature key is masked'
                for b, (ks, chans, vals) in enumerate(singles):
                    m = e[b][:, chans]                                     # (Q, keys) fp16(me[q, c_key])
                    prod = m * vals                                        # exact
                    ok = (m.abs() >= FP16_MIN_NORMAL) | (m == 0)
                    exp_bits = prod <= MASKED_LOGIT_MAX
                    bad = (bits[b][:, ks] != exp_bits) & ok
                    assert not bad.any(), '%s image %d: %d planted bits differ' % (what, b, int(bad.sum()))
                    n_above += int((ok & (prod < 0) & ~exp_bits).sum())
                    n_below += int((ok & exp_bits & (prod > -2 * FP16_MIN_NORMAL)).sum())
                # ---- constant image
                v = _bf16_randn(g, (B, C)).float()
                v[v.abs() < FP16_MIN_NORMAL] = 0                        # fp16(v) == v
                mfc = v[:, :, None, None].expand(B, C, st.H4, st.W4).bfloat16().contiguous()
                _, _, _, _, bm, am = st.rt.head_call(x, mfc.to(DEV), level)
                bits = _check_bits(st, level, bm, am)
                pop = bits.sum(-1)
                assert bool(((pop == 0) | (pop == K)).all()), what + ': constant image, a row is not uniform'
                lg = torch.matmul(e, v.double()[:, :, None])[..., 0]
                clear = (lg - MASKED_LOGIT_MAX).abs() > 2.0 ** -14 * torch.matmul(e.abs(), v.double().abs()[:, :, None])[..., 0]
                assert torch.equal(am.cpu().bool()[clear], (lg <= MASKED_LOGIT_MAX)[clear]), what + ': constant image'
            # both sides of the cut-off were planted: small negative logits that are NOT masked (a sign test would mask
            # them) and masked ones
            assert n_above > 0 and n_below > 0, (n_above, n_below)


# --------------------------------------------------------------------------------------------- K4, exact
@pytest.mark.parametrize('H,W', [(1056, 800), (352, 288), (256, 256)])
def test_k4_kv_projection_exact(H, W):
    """K4 with integer operands: the K and V rows of every layer's cross_in_w in {-1, 0, 1}, level_embed in {-1, 0, 1},
    the key and value biases small integers, memories in {-1, 0, 1} (1 in 8 nonzero).  The bf16 casts and every sum are
    exact, so the K half must EQUAL mem Wk^T (no bias: the key bias reaches the scores as Q R^T in the attention kernel)
    and the V half mem Wv^T + level_embed Wv^T + bv, for every layer slot at every level.  1056x800: 825 keys at level
    0 (re-pitched for TMA; 7 tiles, so the rank-1 CTA of the last pair lies wholly past the end); 352x288: 99 keys at
    level 0 (one pair, its second tile past the end).  B = 3, so a store clipped in the wrong dimension lands in the
    next image's rows, which are pre-filled with NaN."""
    Q, B = 100, 3
    g = torch.Generator().manual_seed(H + W)

    def ints(shape, lo, hi, density=1.0):
        v = torch.randint(lo, hi + 1, shape, generator=g).float()
        return v * (torch.rand(shape, generator=g) < density) if density < 1 else v

    sd = synth.make_params(seed=9, num_queries=Q, perturb=True)
    for i in range(L):
        p = 'transformer_decoder.layers.%d.attentions.0.attn.' % i
        sd[p + 'in_proj_weight'][C:] = ints((2 * C, C), -1, 1)
        sd[p + 'in_proj_bias'][C:] = ints((2 * C,), -4, 4)
    sd['level_embed.weight'] = ints((3, C), -1, 1, 0.125)
    head = _head(Q, sd=sd)
    st = _Stage(head, H, W, B)
    mems = [ints((B, C) + s, -1, 1, 0.125).bfloat16() for s in st.sizes]
    for level in range(3):
        st.kv(level).view(torch.int16).fill_(NAN16)
    st.rt.kv_project([m.to(DEV) for m in mems])
    for level in range(3):
        K = st.K[level]
        got = st.kv(level).cpu().double()
        mk = mems[level].double().view(B, C, K).transpose(1, 2)
        for sl in range(NL):
            p = 'transformer_decoder.layers.%d.attentions.0.attn.' % (sl * 3 + level)
            w, bias = sd[p + 'in_proj_weight'].double(), sd[p + 'in_proj_bias'].double()
            wk, wv, bv = w[C:2 * C], w[2 * C:], bias[2 * C:]
            k_ref = mk @ wk.t()
            v_ref = mk @ wv.t() + (sd['level_embed.weight'][level].double() @ wv.t() + bv)
            assert max(float(k_ref.abs().max()), float(v_ref.abs().max())) <= 256     # exact in bf16
            k_got, v_got = got[:, :, sl * C:(sl + 1) * C], got[:, :, (NL + sl) * C:(NL + sl + 1) * C]
            assert torch.equal(k_got, k_ref), 'level %d slot %d K: %d differ' % (level, sl, int((k_got != k_ref).sum()))
            assert torch.equal(v_got, v_ref), 'level %d slot %d V: %d differ' % (level, sl, int((v_got != v_ref).sum()))


# ------------------------------------------------------------------------------------------------ K1 heads
EPS_K1 = 2.0 ** -14           # split operands 3 * 2^-18 (= 2^-16.4) + fp32 accumulation of 768 terms (768 * 2^-24 = 2^-14.4)
# Relative RMS error (RMS(got - ref) / RMS(ref)) of a correct run on a B200 (1000 W power limit), at Q = 100 and 300:
# cls 4.3e-6, emb 4.3e-6, me 7.4e-6.  The bars are about 4x that; a dropped or misaligned hi/lo term costs ~2^-9.
K1_RMS_BAR = {'cls': 1.7e-5, 'emb': 1.7e-5, 'me': 3e-5}


@pytest.mark.parametrize('Q,ncls1', [(100, 49), (300, 118)])
def test_k1_query_heads_within_propagated_bound(Q, ncls1):
    """K1 (post_norm, then [v2l_transform | mask_embed.0 | cls_embed] and mask_embed.2 / .4 on hi/lo bf16 operand pairs
    with 3 MMAs per product) against fp64.  Elementwise bound, propagated layer by layer:
      z:   dz = 2^-16 (|w| (|x_hat| + 1) + |b|) for the fp32 LayerNorm (its error is a few 2^-24 of those terms),
      out: d_out = |W| d_in + EPS_K1 |W| (|h_in| + d_in) + 2^-22 |out| (bias add), ReLU passing it through.
    The worst case alone cannot see a lost hi/lo term under random signs, so the relative RMS error of each output is
    also held to K1_RMS_BAR."""
    sd = synth.make_params(seed=17, num_queries=Q, perturb=True, num_classes_p1=ncls1)
    head = _head(Q, ncls1=ncls1, sd=sd)
    assert head.use_class_emb
    B = 2
    st = _Stage(head, 256, 256, B)
    g = torch.Generator().manual_seed(Q)
    x = torch.randn((B, Q, C), generator=g)
    cls, emb, _, me, _, _ = st.rt.head_call(x.to(DEV), _bf16_randn(g, (B, C, st.H4, st.W4)).to(DEV), 0, want_bits=False)
    d = lambda k: sd[k].double()
    xd = x.double()
    mu = xd.mean(-1, keepdim=True)
    xh = (xd - mu) / torch.sqrt(((xd - mu) ** 2).mean(-1, keepdim=True) + 1e-5)
    wn, bn = d('transformer_decoder.post_norm.weight'), d('transformer_decoder.post_norm.bias')
    z = xh * wn + bn
    dz = 2.0 ** -16 * (wn.abs() * (xh.abs() + 1) + bn.abs())

    def lin(h, dh, name, relu=False):
        w, b = d(name + '.weight'), d(name + '.bias')
        out = h @ w.t() + b
        dout = dh @ w.abs().t() + EPS_K1 * ((h.abs() + dh) @ w.abs().t()) + 2.0 ** -22 * out.abs()
        return (out.clamp(min=0) if relu else out), dout

    h1, d1 = lin(z, dz, 'mask_embed.0', True)
    h2, d2 = lin(h1, d1, 'mask_embed.2', True)
    refs = {'cls': lin(z, dz, 'cls_embed'), 'emb': lin(z, dz, 'v2l_transform'), 'me': lin(h2, d2, 'mask_embed.4')}
    for name, got in (('cls', cls), ('emb', emb), ('me', me)):
        ref, bound = refs[name]
        err = got.cpu().double() - ref
        worst = float((err.abs() / bound).max())
        rms = float(err.pow(2).mean().sqrt() / ref.pow(2).mean().sqrt())
        print('K1 Q=%d %s: worst %.3g of the bound, relative RMS error %.3g' % (Q, name, worst, rms))
        assert worst <= 1.0, (name, worst)
        assert rms <= K1_RMS_BAR[name], (name, rms)
