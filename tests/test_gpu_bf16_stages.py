"""Stage tests of the bf16 (tcgen05) head call: each GEMM stage against a reference of its OWN arithmetic, in fp64 on
the CPU, at the shapes where the kernels change route.  The end-to-end tests of test_gpu_bf16.py hold the product to
BASELINE's statistical bars (1e-2 of range, 99.9 % of the attention-mask bits); here the bars come from the rounding
steps of each stage, so a dropped term, a wrong row offset or a wrong rounding mode fails although the product bars
would still pass.

  K1  query heads        post_norm -> [v2l | mask_embed.0 | cls] -> mask_embed.2 -> .4, hi/lo bf16 operand pairs
  K2  mask einsum        mask[call, b, q, p] = sum_c bf16(me)[b, call, q, c] mf[b, c, p]            (bf16 output)
  K3  attention-mask     bit = sum_c fp16(me)[b, q, c] fds_l[b, c, key] <= MASKED_LOGIT_MAX            (fp32 accumulate)
  K4  K/V projection     kv_l[b, key, :] = mem_l[b, :, key] [Wk; Wv]^T (+ level_embed Wv^T + bv on V)   (bf16 output)
  K5  cross-attention    out[b, q, h] = softmax_k(bf16(q) . (k + R_layer) | mask) v, R the key-bias table of the layer,
                         K / V the layer slot's column views of kv_l                     (fp32 and IEEE-half output)
  K6  self-attention     the same kernel on K, V interleaved in one (B, Q, 2C) buffer, K = Q, no mask, no table

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


# ------------------------------------------------------------------------------------------------- K5 / K6 attention
# K5 (cross-attention, cgg_masked_attention with `layer`: the handle's key-bias table, IEEE-half rows, K and V as the
# column views of kv_l that tc_decoder_layer passes) and the K6 self-attention form (K and V interleaved in one
# (B, Q, 2C) buffer, no bitmap) against tests/golden/attention_ref.py: exact on constructed scores (every score 0: a
# masked mean; +-1 key codes: one-hot), elsewhere within the rounding bound of attention_ref.reference.
import attention_ref as AR                       # noqa: E402
from cgg_b200 import lib as _clib                 # noqa: E402
from oracle import cgg_oracle as O               # noqa: E402

# Relative RMS error (RMS(got - ref) / RMS(ref)) of the fp32 output, the largest over the cases of each kind in a
# correct run on a B200 (1000 W power limit): production cross-attention ('prod') and random keys ('rand') at each q
# scale, the score ramps and the two-level scores.  The bars are about 4x those values.
K5_RMS_MEASURED = {('prod', 0.25): 6.0e-4, ('prod', 1.0): 7.6e-4, ('prod', 16.0): 3.0e-4,
                   ('rand', 0.25): 1.6e-3, ('rand', 1.0): 9.4e-4, ('rand', 16.0): 2.4e-4,
                   'ramp': 1.15e-3, 'two': 2.1e-3}
K5_RMS_BAR = {key: 4 * val for key, val in K5_RMS_MEASURED.items()}


def _attn_rt(Q, B, H=256, W=256, sd=None):
    head = _head(Q, seed=1, sd=sd)
    return _Stage(head, H, W, B)


def _bits(masked, offset):
    """bitmap (B, Q, W32) int32 on the device; offset: a view one word into its buffer (a misaligned base)."""
    words = O.pack_mask_bits(masked)
    if not offset:
        return words.to(DEV)
    buf = torch.zeros(words.numel() + 1, dtype=torch.int32)
    buf[1:] = words.flatten()
    return buf.to(DEV)[1:].view(words.shape)


def _nan_kv(k, v):
    """k, v (B, K, C) as column views of a NaN-filled (B, K, 4C) bf16 buffer: columns the call must not read are NaN."""
    B, K, _ = k.shape
    buf = torch.full((B, K, 4 * C), NAN16, dtype=torch.int16).view(torch.bfloat16)
    buf[:, :, C:2 * C] = k.bfloat16()
    buf[:, :, 3 * C:] = v.bfloat16()
    buf = buf.to(DEV)
    return buf[:, :, C:2 * C], buf[:, :, 3 * C:]


def _attend(rt, q, k, v, masked=None, am=None, layer=-1, offset=False):
    """Runs the attention twice (bit-identical, and out_half == fp16(out)) and, at B = 3, image 1 alone (bit-identical
    to its rows of the batch).  k, v: device views.  Returns (out, out_half) on the CPU."""
    qd = q.to(DEV)
    bm = _bits(masked, offset) if masked is not None else None
    amd = am.to(torch.uint8).to(DEV) if am is not None else None
    runs = [rt.masked_attention(qd, k, v, bm, amd, layer=layer, out_half=True) for _ in range(2)]
    out, half = runs[0][0].cpu(), runs[0][1].cpu()
    assert torch.equal(out.view(torch.int32), runs[1][0].cpu().view(torch.int32)), 'two runs differ (fp32)'
    assert torch.equal(half.view(torch.int16), runs[1][1].cpu().view(torch.int16)), 'two runs differ (half)'
    assert torch.equal(half.view(torch.int16), out.half().view(torch.int16)), 'out_half != fp16(out)'
    if q.shape[0] == 3:
        one = lambda t: t[1:2] if t is not None else None
        o1, h1 = rt.masked_attention(qd[1:2], k[1:2], v[1:2], one(bm), one(amd), layer=layer, out_half=True)
        assert torch.equal(o1.cpu().view(torch.int32), out[1:2].view(torch.int32)), 'image alone != image in a batch'
        assert torch.equal(h1.cpu().view(torch.int16), half[1:2].view(torch.int16)), 'image alone != image in a batch'
    return out, half


def _check_bound(what, out, half, ref, bound, rms_bar=None):
    for name, got in (('fp32', out), ('half', half)):
        err = (got.double() - ref).abs()
        bad = err > bound
        if bad.any():
            b, qi, c = [int(x) for x in bad.nonzero()[0]]
            raise AssertionError('%s %s: %d outputs outside the bound, first at image %d row %d head %d channel %d: got '
                                 '%.9g want %.9g bound %.3g' % (what, name, int(bad.sum()), b, qi, c // 32, c % 32,
                                                                float(got[b, qi, c]), float(ref[b, qi, c]),
                                                                float(bound[b, qi, c])))
    rms = float((out.double() - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt().clamp(min=1e-300))
    worst = float(((out.double() - ref).abs() / bound.clamp(min=1e-300)).max())
    print('K5 %s: worst %.3g of the bound, relative RMS error %.3g' % (what, worst, rms))
    if rms_bar is not None:
        assert rms <= rms_bar, '%s: relative RMS error %.3g above the bar %.3g' % (what, rms, rms_bar)


def _live_mask(g, B, Q, K, counts):
    """Rows of query tile qt of image b allow keys (density 1/2) only inside n = counts[(b * nqt + qt) % len] chosen
    key tiles, so that exactly n tiles are live for that CTA (0: every row wholly masked)."""
    nt, nqt = (K + AR.KT - 1) // AR.KT, (Q + 127) // 128
    masked = torch.ones((B, Q, K), dtype=torch.bool)
    for b in range(B):
        for qt in range(nqt):
            n = counts[(b * nqt + qt) % len(counts)]
            tiles = torch.randperm(nt, generator=g)[:n]
            rows = slice(qt * 128, min(Q, qt * 128 + 128))
            for t in tiles.tolist():
                cols = slice(t * AR.KT, min(K, t * AR.KT + AR.KT))
                blk = masked[b, rows, cols]
                blk[:] = torch.rand(blk.shape, generator=g) < 0.5
                blk[:, 0] = False                     # the tile is live for every row
    return masked


LIVE_COUNTS = (0, 1, 2, 3, 4, 6, 7)
# (Q, B, K, mask): 1..4 query tiles with rows >= Q in the last; the key tail inside a word and in a new word; 1..3 key
# tiles (fewer than the three score buffers); the 6-stage ring boundary (769 keys = 7 tiles); 512 tiles at 65536 keys.
# 'live': exactly LIVE_COUNTS live tiles per CTA among 32 or more; 'blob': windows; the masks with a '+' run the
# bitmap's word path on a base one word off the alignment (W32 % 4 == 0 takes the vector path otherwise).
K5_EXACT_CASES = [(8, 3, 1, 'rand'), (8, 3, 31, 'rand'), (100, 3, 33, 'rand+'), (100, 3, 64, 'rand'),
                  (100, 3, 99, 'rand'), (128, 3, 128, 'rand+'), (129, 3, 129, 'rand'), (129, 1, 383, 'blob'),
                  (300, 3, 385, 'rand'), (300, 1, 768, 'rand'), (512, 1, 769, 'rand'), (100, 3, 825, 'rand+'),
                  (512, 3, 4096, 'live'), (129, 3, 4096, 'live+'), (100, 1, 16384, 'blob'), (8, 1, 65536, 'rand'),
                  (100, 1, 65536, 'blob+')]


@pytest.mark.parametrize('Q,B,K,kind', K5_EXACT_CASES)
def test_k5_exact_masked_mean(Q, B, K, kind):
    """Case a: q = 0, so every score is 0 and every allowed key has P = exp2(0) = 1; l is the count of allowed keys, O
    an exact integer sum of V in [-8, 8] (< 2^24), and no rescale happens.  out must EQUAL f32(sum) * f32(1 / l) (IEEE
    division, no fast math), out_half fp16 of that, and a row without an allowed key (a full bitmap row without the
    all-masked flag; with 'live' whole CTAs of them: no live tile) zeros.  One wrong mask bit, tail bit, live-tile
    flag, fallback row or quarter merge changes a count or a sum.  Relies on ex2.approx giving exactly 1 at 0 and 0 at
    -inf.  Also at 396 keys with layer 4's key-bias table: q = 0 makes the table's term 0 as well."""
    st = _attn_rt(Q, B)
    g = torch.Generator().manual_seed(Q * 7 + K)
    base = kind.rstrip('+')
    if base == 'live':
        masked, am = _live_mask(g, B, Q, K, LIVE_COUNTS), None
    else:
        masked = AR.random_mask(g, B, Q, K, 0.9 if base == 'blob' else 0.5, blob=base == 'blob')
        am = masked.all(-1)
        am[B - 1, Q - 1] = False                           # a wholly masked row without the flag: no allowed key
        masked[B - 1, Q - 1] = True
    allowed = AR.effective_allowed(masked, am).double()
    k = AR.bf16(torch.randn((B, K, C), generator=g))
    v = torch.randint(-8, 9, (B, K, C), generator=g).float()
    kd, vd = _nan_kv(k, v)
    out, half = _attend(st.rt, torch.zeros((B, Q, C)), kd, vd, masked, am, offset=kind.endswith('+'))
    cnt = allowed.sum(-1, keepdim=True).numpy().astype(np.float32)
    sums = (allowed @ v.double()).numpy().astype(np.float32)
    with np.errstate(divide='ignore'):
        inv = np.where(cnt > 0, np.float32(1) / cnt, np.float32(0)).astype(np.float32)
    want = torch.from_numpy(sums * inv)
    assert not out.isnan().any(), 'NaN in the output'
    bad = out != want
    assert not bad.any(), '%d outputs differ, first at %s' % (int(bad.sum()), bad.nonzero()[0].tolist())
    assert torch.equal(half.view(torch.int16), want.half().view(torch.int16))


def test_k5_exact_masked_mean_with_table():
    B, Q, H, W, layer = 3, 100, 352, 288, 4
    st = _attn_rt(Q, B, H, W)
    K = st.K[layer % 3]
    g = torch.Generator().manual_seed(4)
    masked = AR.random_mask(g, B, Q, K, 0.5)
    am = masked.all(-1)
    v = torch.randint(-8, 9, (B, K, C), generator=g).float()
    kd, vd = _nan_kv(AR.bf16(torch.randn((B, K, C), generator=g)), v)
    out, half = _attend(st.rt, torch.zeros((B, Q, C)), kd, vd, masked, am, layer=layer)
    allowed = AR.effective_allowed(masked, am).double()
    cnt = allowed.sum(-1, keepdim=True).numpy().astype(np.float32)
    want = torch.from_numpy((allowed @ v.double()).numpy().astype(np.float32) * (np.float32(1) / cnt))
    assert torch.equal(out, want), int((out != want).sum())


ALPHA = 64.0


def _codes(K, heads_perm):
    """(K, C) key rows of +-1 codes: per head, bits of the key index in channels 0..15 and bits of a permuted index
    (k * a + c mod 2^16, a odd) in channels 16..31."""
    idx = torch.arange(K)
    bits = lambda x: ((x[:, None] >> torch.arange(16)) & 1).float() * 2 - 1
    rows = []
    for a, c in heads_perm:
        rows += [bits(idx), bits((idx * a + c) % 65536)]
    return torch.cat(rows, 1)


def _one_hot_case(g, B, Q, K):
    """Key codes, V of bf16 normals with 2^-6 <= |v| < 16 (exact in half), a random mask, q = ALPHA x the code of an
    allowed key t per (row, head), so t wins by >= 2 ALPHA = 128 (184 log2 units: every other P flushes to 0).  Every
    4th row instead takes q = ALPHA x [code1(m), 0] of a MASKED key m: its one allowed distance-1 neighbour t wins by
    2 ALPHA, the other neighbours are masked, so a lost mask bit returns v_m or a 50/50 blend.  Row (0, 0) is a
    fallback row (q = the code of any key).  Returns q, k, v, masked, all_masked, t (B, Q, heads)."""
    perm = [(2 * int(torch.randint(1, 30000, (1,), generator=g)) + 1, int(torch.randint(0, 65536, (1,), generator=g)))
            for _ in range(8)]
    k = _codes(K, perm)[None].expand(B, K, C).contiguous()
    e = torch.randint(-6, 4, (B, K, C), generator=g).double()
    mant = 1 + torch.randint(0, 128, (B, K, C), generator=g).double() / 128
    sign = torch.randint(0, 2, (B, K, C), generator=g).double() * 2 - 1
    v = (sign * mant * 2 ** e).float()
    masked = torch.rand((B, Q, K), generator=g) < 0.5
    am = torch.zeros((B, Q), dtype=torch.bool)
    q = torch.zeros((B, Q, C))
    t = torch.zeros((B, Q, 8), dtype=torch.long)
    for b in range(B):
        for qi in range(Q):
            row = masked[b, qi]
            if b == 0 and qi == 0:
                row[:] = True
                am[b, qi] = True
            if qi % 4 == 3 and K > 1:
                m = int(torch.randint(0, K, (1,), generator=g))
                nb = [m ^ (1 << j) for j in range(16) if m ^ (1 << j) < K]
                tt = nb[int(torch.randint(0, len(nb), (1,), generator=g))]
                row[m] = True
                row[nb] = True
                row[tt] = False
                for h in range(8):
                    q[b, qi, h * 32:h * 32 + 16] = ALPHA * k[0, m, h * 32:h * 32 + 16]
                t[b, qi] = tt
                continue
            if not (~row).any():
                row[int(torch.randint(0, K, (1,), generator=g))] = False
            ok = (~row).nonzero()[:, 0] if not am[b, qi] else torch.arange(K)
            for h in range(8):
                tt = int(ok[int(torch.randint(0, len(ok), (1,), generator=g))])
                q[b, qi, h * 32:(h + 1) * 32] = ALPHA * k[0, tt, h * 32:(h + 1) * 32]
                t[b, qi, h] = tt
    return q, k, v, masked, am, t


def _check_one_hot(what, out, half, v, t):
    B, Q, _ = out.shape
    idx = t.repeat_interleave(32, -1)                                 # (B, Q, C): key of each output channel
    want = torch.gather(v, 1, idx)
    bad = half.view(torch.int16) != want.half().view(torch.int16)
    assert not bad.any(), '%s: %d half outputs are not the winning key\'s V, first at %s' % (
        what, int(bad.sum()), bad.nonzero()[0].tolist())
    err = float(((out.double() - want.double()).abs() / want.double().abs()).max())
    assert err <= 2.0 ** -13, (what, err)


@pytest.mark.parametrize('Q,B,K', [(8, 3, 2), (100, 3, 99), (129, 3, 777), (300, 1, 4096), (8, 1, 65536)])
def test_k5_one_hot_exact(Q, B, K):
    """Case b without a table: out_half must equal fp16(v_t) of the winning key t bit for bit, out within 2^-13 |v_t|
    (the fp32 rounding residual of s_t log2e at s_t = 2048 leaves p_t = 2^(+-2^-13) in l)."""
    st = _attn_rt(Q, B)
    g = torch.Generator().manual_seed(K + Q)
    q, k, v, masked, am, t = _one_hot_case(g, B, Q, K)
    kd, vd = _nan_kv(k, v)
    out, half = _attend(st.rt, q, kd, vd, masked, am)
    _check_one_hot('Q=%d B=%d K=%d' % (Q, B, K), out, half, v, t)


@pytest.mark.parametrize('H,W', [(352, 288), (1056, 800)])
def test_k5_one_hot_exact_with_table(H, W):
    """Case b with the production key-bias table of every layer (every level and slot): the cross-attention K weights
    and key bias of the state dict are scaled by 2^-10, and the fp64 table must keep |q . R| <= ALPHA / 4, so that
    the winner still wins by >= 96 (138 log2 units)."""
    Q, B = 100, 3
    sd = synth.make_params(seed=1, num_queries=Q, perturb=True)
    for i in range(L):
        p = 'transformer_decoder.layers.%d.attentions.0.attn.' % i
        sd[p + 'in_proj_weight'][C:2 * C] *= 2.0 ** -10
        sd[p + 'in_proj_bias'][C:2 * C] *= 2.0 ** -10
    st = _attn_rt(Q, B, H, W, sd=sd)
    g = torch.Generator().manual_seed(H)
    for layer in range(L):
        level = layer % 3
        K = st.K[level]
        r, _ = AR.key_bias_table(sd, layer, *st.sizes[level])
        assert float(ALPHA * r.abs().view(K, 8, 32).sum(-1).max()) <= ALPHA / 4
        q, k, v, masked, am, t = _one_hot_case(g, B, Q, K)
        kd, vd = _nan_kv(k, v)
        out, half = _attend(st.rt, q, kd, vd, masked, am, layer=layer)
        _check_one_hot('%dx%d layer %d' % (H, W, layer), out, half, v, t)


def _kv_views(st, level, sl):
    """The production K, V views of layer slot sl in kv_l; every other column (the other slots' K and V) is NaN."""
    buf = st.kv(level)
    keep = torch.zeros(NL * 2 * C, dtype=torch.bool)
    keep[sl * C:(sl + 1) * C] = True
    keep[(NL + sl) * C:(NL + sl + 1) * C] = True
    buf[:, :, ~keep.to(DEV)] = float('nan')
    return buf[:, :, sl * C:(sl + 1) * C], buf[:, :, (NL + sl) * C:(NL + sl + 1) * C]


Q_SCALES = (0.25, 1.0, 16.0)


@pytest.mark.parametrize('H,W,layers', [(352, 288, tuple(range(L))), (1056, 800, (0, 4, 8))])
def test_k5_production_cross_attention_within_bound(H, W, layers):
    """Case c: K and V from cgg_kv_project of random bf16 memories with the synth weights, read as the column views
    that tc_decoder_layer passes (every other column NaN), the handle's key-bias table of the layer, random / blob /
    fallback masks, q at three scales.  Bound: attention_ref.reference against R = (pos + level_embed) Wk^T + bk in
    fp64, plus the RMS bar.  At the sharpest scale the test first shows that the bound can fail: references with the
    table's bf16 hi part only, the neighbouring slot's table and no table each exceed it somewhere."""
    Q, B = 100, 3
    sd = synth.make_params(seed=21, num_queries=Q, perturb=True)
    st = _attn_rt(Q, B, H, W, sd=sd)
    g = torch.Generator().manual_seed(W)
    mems = [_bf16_randn(g, (B, C) + s) for s in st.sizes]
    for layer in layers:
        level, sl = layer % 3, layer // 3
        K = st.K[level]
        st.rt.kv_project([m.to(DEV) for m in mems])
        kv = st.kv(level).cpu()
        k, v = kv[:, :, sl * C:(sl + 1) * C].float(), kv[:, :, (NL + sl) * C:(NL + sl + 1) * C].float()
        kd, vd = _kv_views(st, level, sl)
        r, r_abs = AR.key_bias_table(sd, layer, *st.sizes[level])
        masked = AR.random_mask(g, B, Q, K, (0.5, 0.9, 0.3)[layer % 3], blob=layer % 2 == 1)
        am = masked.all(-1)
        allowed = AR.effective_allowed(masked, am)
        for sigma in Q_SCALES:
            what = '%dx%d layer %d sigma %g' % (H, W, layer, sigma)
            q = torch.randn((B, Q, C), generator=g) * sigma
            ref, bound, _ = AR.reference(q, k, v, allowed, r=r, r_abs=r_abs, half=True)
            if sigma == Q_SCALES[-1]:
                nbr = layer + 3 if layer + 3 < L else layer - 3
                for name, rm in (('hi only', AR.split_hi_lo(r)[0]), ('neighbouring slot', AR.key_bias_table(sd, nbr, *st.sizes[level])[0]),
                                 ('no table', None)):
                    refm = AR.reference(q, k, v, allowed, r=rm)[0]
                    assert bool(((refm - ref).abs() > bound).any()), '%s: the %s reference is within the bound' % (what, name)
            out, half = _attend(st.rt, q, kd, vd, masked, am, layer=layer)
            _check_bound(what, out, half, ref, bound, K5_RMS_BAR[('prod', sigma)])


# the (K, density, blob) cases of the former fp32-output stage test, then score ramps through one channel of K
@pytest.mark.parametrize('case', [('rand', 64, 0.5, False), ('rand', 128, 0.0, False), ('rand', 777, 0.9, False),
                                  ('rand', 4096, 0.5, False), ('rand', 4096, 0.9, True), ('rand', 16384, 0.5, True),
                                  ('ramp', 4096, 10.0, False), ('ramp', 4096, -10.0, False), ('ramp', 1000, 7.5, False),
                                  ('two', 1000, 0.3, False), ('two', 4096, 0.5, True)], ids=str)
def test_k5_random_keys_within_bound(case):
    """Cases c (no table: random bf16 K, V at q scales 0.25 / 1 / 16) and d (attention_ref.ramp_case: the lazy rescale
    with 0 < sc < 2^-8 on every tile, never after the first, and P up to 2^7.5 before a move) and the two-level case
    (attention_ref.two_level_case: exact scores, so the output also must match the float32 emulation within 2^-16 of
    sum p |v| / l; a truncated P is off by 2^-8)."""
    kind, K, density, blob = case
    Q, B = 129, 3
    st = _attn_rt(Q, B)
    g = torch.Generator().manual_seed(K + int(density * 10))
    keep = AR.TWO_LEVEL_ANCHORS if kind == 'two' else ()
    masked = AR.random_mask(g, B, Q, K, density, blob=blob, keep=keep)
    am = masked.all(-1)
    allowed = AR.effective_allowed(masked, am)
    if kind == 'rand':
        k, v = _bf16_randn(g, (B, K, C)).float(), _bf16_randn(g, (B, K, C)).float()
        qs = [(torch.randn((B, Q, C), generator=g) * s, s) for s in Q_SCALES]
    elif kind == 'ramp':
        q, k, v = AR.ramp_case(g, B, Q, K, density)
        qs = [(q, 'ramp')]
    else:
        q, k, v = AR.two_level_case(g, B, Q, K)
        qs = [(q, 'two')]
    kd, vd = _nan_kv(k, v)
    for q, bar in qs:
        what = '%s K=%d %s' % (kind, K, bar)
        ref, bound, _ = AR.reference(q, k, v, allowed, half=True)
        out, half = _attend(st.rt, q, kd, vd, masked, am)
        _check_bound(what, out, half, ref, bound, K5_RMS_BAR[('rand', bar) if kind == 'rand' else bar])
        if kind == 'two':
            emu = AR.emulate(q, k, v, allowed)[0]
            a = AR.reference(q, k, v.abs(), allowed)[0]
            err = float(((out.double() - emu.double()).abs() / a.clamp(min=1e-300)).max())
            assert err <= 2.0 ** -16, (what, err)


@pytest.mark.parametrize('Q', [100, 300])
def test_k6_self_attention_form(Q):
    """Case e: the decoder layer's self-attention call -- K and V interleaved in one buffer (row stride 2C plus 64
    NaN padding columns, image stride Q rows), K = Q keys, no bitmap, half output -- with cases a (q = 0: column means,
    exact), b (one-hot) and c (random, within the bound)."""
    B = 3
    st = _attn_rt(Q, B)
    g = torch.Generator().manual_seed(Q)
    W2 = 2 * C + 64

    def interleaved(k, v):
        buf = torch.full((B, Q, W2), NAN16, dtype=torch.int16).view(torch.bfloat16)
        buf[:, :, :C], buf[:, :, C:2 * C] = k.bfloat16(), v.bfloat16()
        buf = buf.to(DEV)
        return buf[:, :, :C], buf[:, :, C:2 * C]

    # a: every score 0
    v = torch.randint(-8, 9, (B, Q, C), generator=g).float()
    kd, vd = interleaved(AR.bf16(torch.randn((B, Q, C), generator=g)), v)
    out, half = _attend(st.rt, torch.zeros((B, Q, C)), kd, vd)
    want = torch.from_numpy(v.double().sum(1, keepdim=True).numpy().astype(np.float32) * (np.float32(1) / np.float32(Q)))
    assert torch.equal(out, want.expand(B, Q, C)), int((out != want).sum())
    # b: one-hot over Q keys, no mask
    q, k, v, _, _, t = _one_hot_case(g, B, Q, Q)
    for b in range(B):                     # without a bitmap every key is allowed: winners of the unmasked case
        for qi in range(Q):
            for h in range(8):
                q[b, qi, h * 32:(h + 1) * 32] = ALPHA * k[0, t[b, qi, h], h * 32:(h + 1) * 32]
    kd, vd = interleaved(k, v)
    out, half = _attend(st.rt, q, kd, vd)
    _check_one_hot('self-attention Q=%d' % Q, out, half, v, t)
    # c: random operands
    k, v = _bf16_randn(g, (B, Q, C)).float(), _bf16_randn(g, (B, Q, C)).float()
    kd, vd = interleaved(k, v)
    allowed = torch.ones((B, Q, Q), dtype=torch.bool)
    for sigma in Q_SCALES:
        q = torch.randn((B, Q, C), generator=g) * sigma
        ref, bound, _ = AR.reference(q, k, v, allowed, half=True)
        out, half = _attend(st.rt, q, kd, vd)
        _check_bound('self-attention Q=%d sigma %g' % (Q, sigma), out, half, ref, bound)


def test_k5_rejected_on_host():
    """Arguments the entry must refuse, each before any launch (the library's launch count does not move)."""
    Q, B, K = 100, 1, 64
    head = _head(Q, seed=1)
    rt = head._runtime(torch.device(DEV, 0))
    lib = rt.lib
    q = torch.zeros((B, Q, C), device=DEV)
    kv = torch.zeros((B, 65537, C), dtype=torch.bfloat16, device=DEV)
    k = kv[:, :K]

    def refused(code, fn):
        n0 = lib.cgg_launch_count()
        with pytest.raises(_clib.CggError, match=code):
            fn()
        assert lib.cgg_launch_count() == n0, code + ': a kernel was launched'

    refused('CGG_ERR_BAD_SHAPE', lambda: rt.masked_attention(q, k, k, layer=0))          # not prepared: no table
    st = _Stage(head, 256, 256, B)
    refused('CGG_ERR_BAD_SHAPE', lambda: rt.masked_attention(q, k, k, layer=L))
    refused('CGG_ERR_BAD_SHAPE', lambda: rt.masked_attention(q, k, k, layer=-2))
    refused('CGG_ERR_BAD_SHAPE', lambda: rt.masked_attention(q, k, k, layer=1))          # level 1 has 256 keys
    refused('CGG_ERR_BAD_SHAPE', lambda: rt.masked_attention(q, kv, kv))                 # 65537 keys: 513 tiles
    rt.masked_attention(q, kv[:, :65536], kv[:, :65536])                                 # 65536 keys: accepted
    rt.masked_attention(q, kv[:, :st.K[0]], kv[:, :st.K[0]], layer=0)

    def no_output():
        _clib.check(lib.cgg_masked_attention(rt.handle, B, K, q.data_ptr(), k.data_ptr(), k.data_ptr(), C, K * C,
                                             None, None, -1, None, None, rt._stream()), rt.handle, 'no output')
    refused('CGG_ERR_NULL', no_output)
    sd = synth.make_params(seed=1, num_queries=Q, perturb=True)
    rt32 = build_head_from_state_dict(sd, Q, 49, 'fp32', DEV)._runtime(torch.device(DEV, 0))
    rt32.prepare(32, 32, [(4, 4), (8, 8), (16, 16)], B)
    k32 = torch.zeros((B, 16, C), device=DEV)
    refused('CGG_ERR_UNSUPPORTED', lambda: rt32.masked_attention(q, k32, k32, layer=0))
    refused('CGG_ERR_UNSUPPORTED', lambda: rt32.masked_attention(q, k32, k32, out_half=True))
