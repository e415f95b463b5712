"""Pins the oracle (oracle/cgg_oracle.py) against outputs of the reference itself:
the committed golden vectors (tests/golden/*.npz, written by make_golden.py from the
unmodified reference head) and, in the build container, the live reference."""
import os

import numpy as np
import pytest
import torch

from oracle import cgg_oracle as O
from oracle import ref_shim
from cgg_b200 import synth
import cases

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TOL = 2e-5   # fp32 CPU, different summation order only


def _load(name):
    return np.load(os.path.join(GOLD, name))


@pytest.mark.parametrize('name', list(cases.HEAD_CASES))
def test_head_matches_golden(name):
    c = cases.HEAD_CASES[name]
    g = _load('head_%s.npz' % name)
    sd, mf, mems = cases.case_tensors(c)
    assert abs(cases.param_checksum(sd) - float(g['param_checksum'])) < 1e-6 * float(g['param_checksum']), \
        'seeded parameter generator drifted from the one that made the fixtures'
    out = O.decoder_forward(sd, mf, mems)
    assert len(out['cls']) == 10
    n_all = 0
    for j in range(10):
        np.testing.assert_allclose(out['cls'][j].numpy(), g['cls_%d' % j], atol=TOL, rtol=0)
        emb = out['emb'][j].numpy()
        np.testing.assert_allclose(emb if j in (0, 4, 9) else emb[:, :, ::16], g['emb_%d' % j], atol=TOL, rtol=0)
        flat = out['mask'][j].flatten()[::cases.MASK_SAMPLE_STRIDE].numpy()
        np.testing.assert_allclose(flat, g['mask_sample_%d' % j], atol=5e-5, rtol=0)
        assert abs(float(out['mask'][j].double().abs().sum()) - float(g['mask_abssum_%d' % j])) \
            < 1e-5 * float(g['mask_abssum_%d' % j])
        bits = O.pack_mask_bits(out['masked'][j]).numpy()
        assert np.array_equal(bits, g['bits_%d' % j]), 'attention-mask bits differ at head call %d' % j
        n_all += int((out['masked'][j].sum(-1) == out['masked'][j].shape[-1]).sum())
    assert n_all == int(g['n_all_masked_rows'])
    np.testing.assert_allclose(out['mask'][9].numpy(), g['last_mask_full'], atol=5e-5, rtol=0)
    if 'cls_emb_logits_9' in g:      # OSPS case: real class embeddings, 118 class rows (head.py:631-648)
        got = O.cls_emb_logits(out['emb'][9], sd['class_embs'], 10.0).numpy()
        np.testing.assert_allclose(got, g['cls_emb_logits_9'], atol=5e-4, rtol=0)


def test_fallback_case_really_hits_fallback():
    assert int(_load('head_dense_fallback.npz')['n_all_masked_rows']) > 10
    assert int(_load('head_tiny.npz')['n_all_masked_rows']) == 0


@pytest.mark.parametrize('name', list(cases.GROUNDING_CASES))
def test_grounding_matches_golden(name):
    g = _load('grounding.npz')
    pred, cap, m = cases.grounding_tensors(name)
    pred.requires_grad_(True)
    loss = O.grounding_loss(pred, cap, m, 10.0, loss_weight=2.0)
    loss.backward()
    assert abs(loss.item() - float(g[name + '_loss'])) < 2e-5 * max(1.0, abs(float(g[name + '_loss'])))
    np.testing.assert_allclose(pred.grad.flatten()[::cases.GRAD_SAMPLE_STRIDE].numpy(),
                               g[name + '_grad_sample'], atol=1e-6, rtol=1e-4)
    assert abs(float(pred.grad.double().abs().sum()) - float(g[name + '_grad_abssum'])) \
        < 1e-4 * float(g[name + '_grad_abssum'])


def test_embedding_side_matches_golden():
    g = _load('embeddings.npz')
    sd = synth.make_params(seed=9, num_queries=16)
    ids, mask, table, _, _ = synth.make_captions(5, 4, vocab=400 + 1000)
    ne = O.noun_embeddings(table, torch.from_numpy(g['ln_w']), torch.from_numpy(g['ln_b']), ids)
    np.testing.assert_allclose(ne.numpy(), g['noun_embs'], atol=2e-5, rtol=0)
    pred = torch.from_numpy(g['pred'])
    np.testing.assert_allclose(O.cls_emb_logits(pred, sd['class_embs'], 10.0).numpy(), g['logits'], atol=2e-4, rtol=0)
    np.testing.assert_allclose(O.test_time_grounding(pred[0], ne[0]).numpy(), g['att'], atol=2e-4, rtol=0)


def test_pos_enc_properties():
    p = O.sine_pos_enc(5, 7)
    assert p.shape == (35, 256)
    # first half depends on the row only, second half on the column only
    p = p.view(5, 7, 256)
    assert torch.equal(p[:, 0, :128], p[:, 3, :128]) and torch.equal(p[0, :, 128:], p[4, :, 128:])
    assert float(p.abs().max()) <= 1.0


def test_mask_threshold_is_not_sign_test():
    """sigmoid(x) < 0.5 in fp32 is true only for x <= -1.7881392e-07 (SURVEY.md section 7.2)."""
    x = torch.tensor([-1e-6, -1.7881393e-07, -1.19e-07, -1e-9, 0.0, 1e-9])[None, None, None, :]
    x = x.expand(1, 1, 1, 6).contiguous()
    m = O.attn_mask_from_logits(x, (1, 6))[0, 0]
    assert m.tolist() == [True, True, False, False, False, False]


def test_bilinear_matches_torch():
    import torch.nn.functional as F
    x = torch.randn(2, 5, 64, 48)
    for hw in [(8, 6), (16, 12), (32, 24)]:
        a = F.interpolate(x, hw, mode='bilinear', align_corners=False)
        b = O.bilinear_resize(x, hw)
        assert float((a - b).abs().max()) < 3e-7
        assert bool(((a.sigmoid() < 0.5) == (b.sigmoid() < 0.5)).all())


def test_level_resample_formula_is_torch_bilinear():
    """The reference of the bf16 path's level resample (test_gpu_bf16_stages.level_resample_ref, the arithmetic of
    downsample3_kernel) is torch's bilinear resize: on bf16-valued inputs, what the pixel decoder hands the head,
    fp16(formula) == fp16(F.interpolate(bilinear, align_corners=False)) bit for bit at the ratios 8, 4 and 2.  The
    comparison is made in fp16, the precision the resampled features are stored in: in fp32, torch's vectorised CPU
    loop rounds a few in 10^6 values one ulp differently at ratios 4 and 8."""
    import torch.nn.functional as F
    from test_gpu_bf16_stages import RATIOS, level_resample_ref
    mf = torch.randn((2, 256, 264, 200), generator=torch.Generator().manual_seed(0)).bfloat16()
    for r in RATIOS:
        want = F.interpolate(mf.float(), (264 // r, 200 // r), mode='bilinear', align_corners=False).half()
        got = level_resample_ref(mf, r).half()
        assert torch.equal(got.view(torch.int16), want.view(torch.int16)), r


def test_pack_bits_layout():
    m = torch.zeros(1, 2, 40, dtype=torch.bool)
    m[0, 0, 0] = m[0, 0, 31] = m[0, 0, 33] = True
    m[0, 1, 39] = True
    w = O.pack_mask_bits(m)
    assert w.shape == (1, 2, 2)
    assert (w[0, 0, 0].item() & 0xffffffff) == 0x80000001 and w[0, 0, 1].item() == 2
    assert w[0, 1, 0].item() == 0 and w[0, 1, 1].item() == 1 << 7


@pytest.mark.skipif(not ref_shim.reference_available(), reason='reference tree only exists in the build container')
def test_oracle_matches_live_reference():
    R = ref_shim.REF_ROOT
    head = ref_shim.build_reference_head(num_queries=24, known_file=R + '/datasets/unknown/known_65.txt',
                                         unknown_file=R + '/datasets/unknown/unknown_17.txt')
    sd = synth.make_params(seed=21, num_queries=24, perturb=True)
    head.load_state_dict(sd, strict=True)
    mf, mems = synth.make_inputs(9, 2, 128, 96)
    ref = ref_shim.run_reference_head(head, mf, mems)
    out = O.decoder_forward(sd, mf, mems)
    for j in range(10):
        assert float((ref[0][j] - out['cls'][j]).abs().max()) < TOL
        assert float((ref[1][j] - out['emb'][j]).abs().max()) < TOL
        assert float((ref[2][j] - out['mask'][j]).abs().max()) < 5e-5


@pytest.mark.skipif(not ref_shim.reference_available(), reason='reference tree only exists in the build container')
def test_oracle_pred_emb_norm_matches_live_reference():
    """head.py:743-744: the optional L2 normalisation of the embedding predictions."""
    R = ref_shim.REF_ROOT
    head = ref_shim.build_reference_head(num_queries=24, known_file=R + '/datasets/unknown/known_65.txt',
                                         unknown_file=R + '/datasets/unknown/unknown_17.txt')
    sd = synth.make_params(seed=22, num_queries=24, perturb=True)
    head.load_state_dict(sd, strict=True)
    head.pred_emb_norm = True
    mf, mems = synth.make_inputs(10, 1, 64, 64)
    ref = ref_shim.run_reference_head(head, mf, mems)
    out = O.decoder_forward(sd, mf, mems, pred_emb_norm=True)
    for j in range(10):
        assert float((ref[1][j] - out['emb'][j]).abs().max()) < TOL
        assert float((out['emb'][j].norm(dim=-1) - 1).abs().max()) < 1e-5



def _bound_ratio(got, ref, bound):
    """max |got - ref| / bound; a nonzero error where the bound is 0 (a row without an allowed key) counts as inf."""
    err = (got.double() - ref).abs()
    r = torch.where(bound > 0, err / bound.clamp(min=1e-300), torch.where(err > 0, float('inf'), 0.0))
    return float(r.max())


def test_attention_bound_passes_the_kernel_emulation_and_fails_its_mutants():
    """The elementwise bound of the bf16 attention kernel (tests/golden/attention_ref.py, used by the K5 GPU tests) on
    a float32 emulation of the kernel's arithmetic: bf16(q), P = bf16(e) with an fp32 l, the per-quarter lazy
    reference, the half store.  The emulation must stay within it, and each mutant -- the table's hi part only, the
    neighbouring slot's table, P truncated to bf16, no rescale (sc = 1), the tail mask ignored, the fallback ignored --
    must exceed it somewhere, so the GPU tests' bound is known to be able to fail.  Production-like inputs: layer 4's
    table (level 1, slot 1) on a 22x18 level (396 keys, a partial last tile)."""
    import attention_ref as A
    g = torch.Generator().manual_seed(0)
    B, Q, C = 2, 64, 256
    sd = synth.make_params(seed=3, num_queries=Q, perturb=True)
    h, w, layer = 22, 18, 4
    K = h * w
    r, r_abs = A.key_bias_table(sd, layer, h, w)
    hi, lo = A.split_hi_lo(r)
    nhi, nlo = A.split_hi_lo(A.key_bias_table(sd, layer + 3, h, w)[0])
    wkv = sd['transformer_decoder.layers.%d.attentions.0.attn.in_proj_weight' % layer][C:]
    mem = torch.randn((B, K, C), generator=g)
    k, v = A.bf16(mem @ wkv[:C].t()), A.bf16(mem @ wkv[C:].t())
    masked = A.random_mask(g, B, Q, K, 0.5)
    am = masked.all(-1)
    allowed = A.effective_allowed(masked, am)
    q = torch.randn((B, Q, C), generator=g) * 16          # sharp: the table's lo part matters
    ref, bound, _ = A.reference(q, k, v, allowed, r=r, r_abs=r_abs, half=True)
    out, half = A.emulate(q, k, v, allowed, hi, lo)
    assert _bound_ratio(out, ref, bound) <= 0.5 and _bound_ratio(half, ref, bound) <= 0.5
    mutants = {'hi only': A.emulate(q, k, v, allowed, hi)[0],
               'neighbouring slot': A.emulate(q, k, v, allowed, nhi, nlo)[0],
               'sc = 1': A.emulate(q, k, v, allowed, hi, lo, mutant='sc_one')[0],
               'tail ignored': A.emulate(q, k, v, allowed, hi, lo, mutant='tail')[0],
               'fallback ignored': A.emulate(q, k, v, A.effective_allowed(masked, None), hi, lo)[0]}
    # P's rounding, on exact two-level scores and positive V (a truncated P is 2^-7.5 low, the bound allows 2^-8)
    K2 = 1000
    q2, k2, v2 = A.two_level_case(g, B, Q, K2)
    al2 = A.effective_allowed(A.random_mask(g, B, Q, K2, 0.3, keep=A.TWO_LEVEL_ANCHORS), None)
    ref2, bound2, _ = A.reference(q2, k2, v2, al2, half=True)
    assert _bound_ratio(A.emulate(q2, k2, v2, al2)[1], ref2, bound2) <= 0.75
    worst = {name: _bound_ratio(got, ref, bound) for name, got in mutants.items()}
    worst['P truncated'] = _bound_ratio(A.emulate(q2, k2, v2, al2, mutant='p_trunc')[0], ref2, bound2)
    assert all(x > 1.1 for x in worst.values()), worst
