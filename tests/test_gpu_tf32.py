"""GPU tests of the tensor-core (tcgen05 kind::tf32) form of cgg_gemm_f32 -- the contraction every linear layer, the mask
einsum (mask2former_head.py:748) and all of their gradients go through in the training step.  Checked against fp64
matmul: exactly on operands that are representable in tf32 (any tile / swizzle / operand-major mistake shows up as a
wrong integer), and within the tf32 rounding bound on random fp32 operands."""
import pytest
import torch

from cgg_b200 import synth
from cgg_b200.head import build_head_from_state_dict
from cgg_b200.train import _K

pytestmark = pytest.mark.gpu
DEV = 'cuda'


@pytest.fixture(scope='module')
def kern():
    sd = synth.make_params(seed=1, num_queries=8)
    head = build_head_from_state_dict(sd, 8, 49, 'fp32', DEV)
    return _K(head._runtime(torch.device(DEV, 0)), tf32=True)


def _operand(rows, K, batch, major, g, ints):
    """(batch, rows, K) logical operand stored K-major ('k') or MN-major ('m'); returns (logical view, strides b/r/k)."""
    shape = (batch, rows, K) if major == 'k' else (batch, K, rows)
    t = torch.randint(-8, 9, shape, generator=g).float() if ints else torch.randn(shape, generator=g)
    t = t.to(DEV)
    if major == 'k':
        return t, t, (rows * K, K, 1)
    return t, t.transpose(1, 2), (rows * K, 1, rows)


CASES = [
    # M, N, K, batch, a_major, b_major, c_mmajor, bias, res, relu, alpha
    (400, 256, 256, 1, 'k', 'k', False, True, False, True, 1.0),          # linear + bias + relu
    (400, 256, 2048, 1, 'k', 'k', False, True, True, False, 0.5),         # FFN2 + residual
    (400, 2048, 256, 1, 'k', 'k', False, True, False, True, 1.0),         # FFN1
    (400, 768, 256, 1, 'k', 'k', False, True, False, False, 1.0),         # v2l_transform
    (400, 256, 2048, 1, 'k', 'm', False, False, False, False, 1.0),       # dX = dY W
    (256, 256, 4100, 1, 'm', 'm', False, False, False, False, 0.176),     # dW = dY^T X, split over K
    (2048, 256, 400, 1, 'm', 'm', False, False, False, False, 1.0),       # dW of FFN1
    (3072, 200, 256, 2, 'm', 'k', True, False, False, False, 1.0),        # mask einsum forward
    (200, 256, 3072, 2, 'k', 'k', False, False, False, False, 1.0),       # d mask_embed, split over K
    (3072, 256, 200, 2, 'm', 'm', True, False, False, False, 1.0),        # d mask_features
    (130, 24, 40, 3, 'k', 'k', False, True, True, False, 2.0),            # ragged edges
    (70, 300, 36, 1, 'm', 'k', False, False, False, False, 1.0),          # N > 256: two column tiles
    (400, 256, 118, 1, 'k', 'm', False, False, False, False, 1.0),        # dX of the 118-class head: SIMT (pitch 472 B)
]


@pytest.mark.parametrize('case', CASES)
@pytest.mark.parametrize('ints', [True, False])
def test_tf32_gemm_against_fp64(kern, case, ints):
    M, N, K, batch, am, bm, c_mmajor, has_bias, has_res, relu, alpha = case
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a_store, a, sA = _operand(M, K, batch, am, g, ints)
    w_store, w, sW = _operand(N, K, batch, bm, g, ints)
    bias = torch.randn(N, generator=g).to(DEV) if has_bias else None
    res = torch.randn((batch, M, N), generator=g).to(DEV) if has_res else None
    if c_mmajor:
        c_store = torch.full((batch, N, M), float('nan'), device=DEV)
        c, sC = c_store.transpose(1, 2), (M * N, 1, M)
    else:
        c_store = torch.full((batch, M, N), float('nan'), device=DEV)
        c, sC = c_store, (M * N, N, 1)
    kern.gemm(a_store, sA, w_store, sW, c_store, sC, M, N, K, batch=batch, bias=bias, R=res, sR=(M * N, N, 1), r_mod=M,
              alpha=alpha, relu=relu, a_mmajor=(am == 'm'), c_mmajor=c_mmajor)
    torch.cuda.synchronize()
    want = torch.matmul(a.double(), w.double().transpose(1, 2))
    if has_bias:
        want = want + bias.double()
    want = want * alpha
    if has_res:
        want = want + res.double()
    if relu:
        want = want.clamp_min(0)
    err = float((c.double() - want).abs().max())
    scale = float(want.abs().max())
    assert torch.isfinite(c).all()
    if ints:
        assert err <= 2e-6 * scale, (err, scale)          # operands exact in tf32: only the fp32 epilogue rounds
    else:
        # 10-bit operand mantissas (truncated): 2 * 2^-10 per product, accumulated over K terms of mixed sign
        bound = 2.0 ** -9 * float((a.double().abs() @ w.double().abs().transpose(1, 2)).max()) * abs(alpha)
        assert err <= bound, (err, bound, scale)
        assert err <= 4e-3 * scale + 1e-3, (err, scale)


def test_tf32_switch_off_is_exact_fp32(kern):
    """tf32 = 0 keeps the parity-mode FMA kernel: fp32 products, error at the fp32 rounding level."""
    k32 = _K(kern.rt, tf32=False)
    g = torch.Generator().manual_seed(5)
    a = torch.randn((300, 256), generator=g).to(DEV)
    w = torch.randn((256, 256), generator=g).to(DEV)
    c = torch.empty((300, 256), device=DEV)
    k32.gemm(a, (0, 256, 1), w, (0, 256, 1), c, (0, 256, 1), 300, 256, 256)
    want = a.double() @ w.double().t()
    assert float((c.double() - want).abs().max()) < 2e-5 * float(want.abs().max())


def test_two_level_batch_matches_fp64(kern):
    """(image, head) batches: item z of A / W / C at (z / inner) * outer stride + (z % inner) * inner stride."""
    B, H, Q, K, d = 2, 8, 40, 96, 32
    Cc = H * d
    g = torch.Generator().manual_seed(11)
    q = torch.randint(-8, 9, (B, Q, Cc), generator=g).float().to(DEV)
    kk = torch.randint(-8, 9, (B, K, Cc), generator=g).float().to(DEV)
    S = torch.full((B, H, Q, K), float('nan'), device=DEV)
    kern.gemm(q, (Q * Cc, Cc, 1), kk, (K * Cc, Cc, 1), S, (H * Q * K, K, 1), Q, K, d, batch=B * H, batch_inner=H,
              s2=(d, d, Q * K))
    want = torch.einsum('bqhd,bkhd->bhqk', q.view(B, Q, H, d).double(), kk.view(B, K, H, d).double())
    assert float((S.double() - want).abs().max()) == 0.0
    # and the transposed product with an MN-major pair: dk[b,key,h,:] = sum_q S[b,h,q,key] q[b,q,h,:]
    dk = torch.full((B, K, Cc), float('nan'), device=DEV)
    Sm = (S / 64).round().clamp(-8, 8)
    kern.gemm(Sm, (H * Q * K, 1, K), q, (Q * Cc, 1, Cc), dk, (K * Cc, Cc, 1), K, d, Q, batch=B * H, batch_inner=H,
              s2=(Q * K, d, d), a_mmajor=True)
    want = torch.einsum('bhqk,bqhd->bkhd', Sm.double(), q.view(B, Q, H, d).double()).reshape(B, K, Cc)
    assert float((dk.double() - want).abs().max()) == 0.0


@pytest.mark.parametrize('Q,K,masked', [(40, 320, True), (24, 20, True), (100, 100, False), (200, 4096, True)])
def test_attention_views_as_tensor_core_products_match_fp32_kernels(kern, Q, K, masked):
    """_AttentionViews (tf32 products + row softmax with the bitmap) on (B, L, 8, 32) views, the decoder's tf32 attention,
    against the flash-style fp32 kernels: forward and the three gradients, including all-masked fallback rows."""
    from cgg_b200.train import _Attention, _AttentionViews
    B, Cc = 2, 256
    g = torch.Generator().manual_seed(Q + K)
    mk = lambda *s: (torch.randn(s, generator=g) * 0.5).to(DEV).requires_grad_(True)
    q, kk, v = mk(B, Q, Cc), mk(B, K, Cc), mk(B, K, Cc)
    bitmap = am = None
    if masked:
        m = torch.rand((B, Q, K), generator=g) < 0.6
        m[0, 1] = True                                       # a fully masked row -> fallback: attends everything
        from oracle import cgg_oracle as O
        bitmap = O.pack_mask_bits(m).to(DEV)
        am = m.all(-1).to(torch.uint8).to(DEV)
    k32 = _K(kern.rt, tf32=False)
    dout = torch.randn((B, Q, Cc), generator=g).to(DEV)
    o_ref = _Attention.apply(k32, q, kk, v, bitmap, am, 8)
    g_ref = torch.autograd.grad(o_ref, (q, kk, v), dout)
    o = _AttentionViews.apply(kern, q.view(B, Q, 8, 32), kk.view(B, K, 8, 32), v.view(B, K, 8, 32), bitmap, am, 1.0)
    g_tc = torch.autograd.grad(o, (q, kk, v), dout)
    torch.cuda.synchronize()
    assert float((o - o_ref).abs().max()) < 5e-3 * float(o_ref.abs().max())
    for a, b_ in zip(g_tc, g_ref):
        assert float((a - b_).abs().max()) < 1e-2 * float(b_.abs().max()), float((a - b_).abs().max()) / float(b_.abs().max())
