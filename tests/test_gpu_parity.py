"""GPU parity tests (run on the B200 box): the CUDA path, called through the C-ABI library,
against the oracle (oracle/cgg_oracle.py, CPU fp32) and the committed golden vectors that came
from the unmodified reference.  fp32 mode: attention-mask bits must be identical; floats within
the tolerances written in each test (different fp32 summation order only)."""
import os

import numpy as np
import pytest
import torch

from oracle import cgg_oracle as O
from cgg_b200 import synth
from cgg_b200.head import build_head_from_state_dict
import cases

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
DEV = 'cuda'


def _bits_np(t):
    return t.cpu().numpy().astype(np.int32)


def _head(sd, q, precision='fp32'):
    return build_head_from_state_dict(sd, q, sd['cls_embed.weight'].shape[0], precision, DEV)


# --------------------------------------------------------------------------------- stages
def test_mask_bits_stage_is_bit_exact():
    """K3 alone: identical logits in -> identical bits out (SURVEY.md section 7 protocol (a))."""
    sd = synth.make_params(seed=1, num_queries=24)
    head = _head(sd, 24)
    g = torch.Generator().manual_seed(5)
    for (H4, W4, th, tw) in [(64, 64, 8, 8), (64, 64, 16, 16), (64, 64, 32, 32), (40, 24, 5, 3), (40, 24, 20, 12),
                             (66, 50, 33, 25)]:
        mp = torch.randn((2, 24, H4, W4), generator=g) * 2.0
        # plant values around the sigmoid<0.5 cutoff (not a sign test) and exact zeros
        planted = torch.tensor([-1e-6, -2.5e-7, -1.0e-7, -1e-9, 0.0, 1e-9, 3e-7])
        s = H4 // th
        for n, v in enumerate(planted):
            r, c = (n % th) * s, ((n * 3) % tw) * s
            mp[0, 1, r:r + s, c:c + s] = v
        mp[1, 3] = -5.0          # a fully masked row -> all_masked flag
        mp[1, 4] = +5.0          # nothing masked
        want = O.attn_mask_from_logits(mp, (th, tw))
        rt = head._runtime(torch.device(DEV, 0))
        rt.prepare(H4, W4, [(th, tw)] * 3, 2)
        bm, am = rt.attn_mask_from_logits(mp.to(DEV), (th, tw))
        assert np.array_equal(_bits_np(bm), O.pack_mask_bits(want).numpy()), (H4, W4, th, tw)
        assert torch.equal(am.cpu().bool(), want.all(-1))
        assert bool(am[1, 3]) and not bool(am[1, 4])
        # and against PyTorch's own CUDA interpolate + sigmoid (the GPU reference order)
        ref = torch.nn.functional.interpolate(mp.to(DEV), (th, tw), mode='bilinear', align_corners=False)
        ref = (ref.sigmoid() < 0.5).flatten(2).cpu()
        assert np.array_equal(_bits_np(bm), O.pack_mask_bits(ref).numpy())


@pytest.mark.parametrize('K,density', [(12, 0.5), (100, 0.0), (777, 0.9), (4096, 0.5), (4096, 0.97)])
def test_masked_attention_stage(K, density):
    """K5 core vs the oracle's softmax(q k^T + mask) v, incl. fallback rows and ragged K."""
    B, Q, C = 2, 24, 256
    sd = synth.make_params(seed=1, num_queries=Q)
    head = _head(sd, Q)
    rt = head._runtime(torch.device(DEV, 0))
    rt.prepare(16, 16, [(2, 2)] * 3, B)
    g = torch.Generator().manual_seed(K)
    q = torch.randn((B, Q, C), generator=g) * 0.4
    k = torch.randn((B, K, C), generator=g)
    v = torch.randn((B, K, C), generator=g)
    masked = torch.rand((B, Q, K), generator=g) < density
    masked[0, 0] = True                      # fully masked row -> fallback (attend everywhere)
    masked[1, 5, : K // 2] = True
    am = masked.all(-1)
    eff = O.apply_fallback(masked)
    s = torch.einsum('bqhd,bkhd->bhqk', q.view(B, Q, 8, 32), k.view(B, K, 8, 32))
    s = s.masked_fill(eff[:, None], float('-inf'))
    want = torch.einsum('bhqk,bkhd->bqhd', torch.softmax(s, -1), v.view(B, K, 8, 32)).reshape(B, Q, C)
    got = rt.masked_attention(q.to(DEV), k.to(DEV), v.to(DEV), O.pack_mask_bits(masked).to(DEV),
                              am.to(torch.uint8).to(DEV))
    assert float((got.cpu() - want).abs().max()) < 2e-5
    if density == 0.0:
        got2 = rt.masked_attention(q.to(DEV), k.to(DEV), v.to(DEV))
        s2 = torch.einsum('bqhd,bkhd->bhqk', q.view(B, Q, 8, 32), k.view(B, K, 8, 32))
        want2 = torch.einsum('bhqk,bkhd->bqhd', torch.softmax(s2, -1), v.view(B, K, 8, 32)).reshape(B, Q, C)
        assert float((got2.cpu() - want2).abs().max()) < 2e-5


# ------------------------------------------------------------------- whole path vs golden
@pytest.mark.parametrize('name', list(cases.HEAD_CASES))
def test_head_fp32_matches_reference_golden(name):
    c = cases.HEAD_CASES[name]
    gold = np.load(os.path.join(GOLD, 'head_%s.npz' % name))
    sd, mf, mems = cases.case_tensors(c)
    head = _head(sd, c['num_queries'])
    cls, emb, mask, dbg = head.decoder_forward(mf.to(DEV), [m.to(DEV) for m in mems], return_debug=True)
    assert len(cls) == len(emb) == len(mask) == 10
    n_all = 0
    for j in range(10):
        np.testing.assert_allclose(cls[j].cpu().numpy(), gold['cls_%d' % j], atol=1e-4, rtol=0)
        e = emb[j].cpu().numpy()
        np.testing.assert_allclose(e if j in (0, 4, 9) else e[:, :, ::16], gold['emb_%d' % j], atol=1e-4, rtol=0)
        np.testing.assert_allclose(mask[j].flatten()[::cases.MASK_SAMPLE_STRIDE].cpu().numpy(),
                                   gold['mask_sample_%d' % j], atol=2e-4, rtol=0)
        if j < 9:
            # boolean attention masks: bit-exact in fp32 mode
            assert np.array_equal(_bits_np(dbg['bitmaps'][j]), gold['bits_%d' % j]), 'mask bits differ at call %d' % j
            n_all += int(dbg['all_masked'][j].sum())
    np.testing.assert_allclose(mask[9].cpu().numpy(), gold['last_mask_full'], atol=2e-4, rtol=0)
    if 'cls_emb_logits_9' in gold:      # OSPS case: 118 class rows, the reference's real class embeddings
        assert tuple(cls[9].shape) == (c['batch'], c['num_queries'], 118)
        np.testing.assert_allclose(head._get_cls_emb_logits(emb[9]).cpu().numpy(), gold['cls_emb_logits_9'],
                                   atol=1e-3, rtol=0)
    if name == 'dense_fallback':
        assert n_all > 10      # the fallback path really ran
        last_rows = int(((gold['bits_9'] != 0).sum()))  # noqa: F841  (bits_9 is never consumed, head.py:841)


def test_teacher_forced_layers_q100():
    """Protocol (b): every layer fed the oracle's decoder state; masks bit-exact except where the
    downsampled logit is within 1e-5 of the threshold, floats within 2e-4."""
    Q, B, H, W = 100, 2, 256, 320
    sd = synth.make_params(seed=11, num_queries=Q, perturb=True)
    mf, mems = synth.make_inputs(4, B, H, W)
    ref = O.decoder_forward(sd, mf, mems)
    head = _head(sd, Q)
    dev = torch.device(DEV, 0)
    rt = head._runtime(dev)
    sizes = [tuple(m.shape[-2:]) for m in mems]
    rt.prepare(mf.shape[2], mf.shape[3], sizes, B)
    mfd = mf.to(dev)
    rt.kv_project([m.to(dev) for m in mems])
    total_bits = flipped = 0
    for i in range(9):
        x = ref['x'][i].to(dev).contiguous()
        cls, emb, mask, me, bm, am = rt.head_call(x, mfd, i % 3)
        assert float((cls.cpu() - ref['cls'][i]).abs().max()) < 2e-4
        assert float((emb.cpu() - ref['emb'][i]).abs().max()) < 2e-4
        assert float((me.cpu() - ref['mask_embed'][i]).abs().max()) < 2e-4
        assert float((mask.cpu() - ref['mask'][i]).abs().max()) < 5e-4
        want_bits = O.pack_mask_bits(ref['masked'][i]).numpy()
        diff = np.bitwise_xor(_bits_np(bm), want_bits)
        nflip = int(np.unpackbits(diff.view(np.uint8)).sum())
        if nflip:
            # every disagreement must sit on the threshold
            d = O.bilinear_resize(ref['mask'][i], sizes[i % 3]).flatten(2)
            got = torch.from_numpy(np.unpackbits(_bits_np(bm).view(np.uint8), bitorder='little')
                                   .reshape(B, Q, -1)[:, :, :d.shape[-1]]).bool()
            bad = got != ref['masked'][i]
            assert float(d[bad].abs().max()) < 1e-5
        flipped += nflip
        total_bits += ref['masked'][i].numel()
        # layer i from the ORACLE's mask (so a threshold-band flip cannot leak into the float check)
        x_out = rt.decoder_layer(i, x, torch.from_numpy(want_bits).to(dev),
                                 ref['masked'][i].all(-1).to(torch.uint8).to(dev))
        assert float((x_out.cpu() - ref['x'][i + 1]).abs().max()) < 3e-4, 'layer %d' % i
    assert flipped <= 2, (flipped, total_bits)


def test_free_running_agreement_q100():
    """Protocol (c): free-running forward; report-level check that outputs stay close."""
    Q, B, H, W = 100, 1, 256, 256
    sd = synth.make_params(seed=12, num_queries=Q, perturb=True)
    mf, mems = synth.make_inputs(5, B, H, W)
    ref = O.decoder_forward(sd, mf, mems)
    head = _head(sd, Q)
    cls, emb, mask, dbg = head.decoder_forward(mf.to(DEV), [m.to(DEV) for m in mems], return_debug=True)
    agree = []
    for j in range(9):
        want = O.pack_mask_bits(ref['masked'][j]).numpy()
        diff = np.bitwise_xor(_bits_np(dbg['bitmaps'][j]), want)
        agree.append(1.0 - np.unpackbits(diff.view(np.uint8)).sum() / ref['masked'][j].numel())
    assert min(agree) > 0.9999, agree
    rng = float(ref['mask'][9].abs().max())
    assert float((mask[9].cpu() - ref['mask'][9]).abs().max()) < 1e-3 * rng


# ---------------------------------------------------------- full size: properties only
def test_full_size_1024_properties():
    """BASELINE config size (1024x1024, Q=100), B=2: size-independent properties --
    (i) the bitmap equals K3 re-applied (by torch CUDA ops) to our own mask logits;
    (ii) the path is per-image independent: image 0 alone gives the same bits/logits as in a batch;
    (iii) determinism: two runs are bitwise identical."""
    Q, B = 100, 2
    sd = synth.make_params(seed=0, num_queries=Q)
    mf, mems = synth.make_inputs(0, B, 1024, 1024)
    head = _head(sd, Q)
    mfd, memd = mf.to(DEV), [m.to(DEV) for m in mems]
    cls, emb, mask, dbg = head.decoder_forward(mfd, memd, return_debug=True)
    sizes = [tuple(m.shape[-2:]) for m in mems]
    for j in range(9):
        d = torch.nn.functional.interpolate(mask[j], sizes[j % 3], mode='bilinear', align_corners=False)
        want = (d.sigmoid() < 0.5).flatten(2).cpu()
        assert np.array_equal(_bits_np(dbg['bitmaps'][j]), O.pack_mask_bits(want).numpy()), j
    cls2, emb2, mask2, dbg2 = head.decoder_forward(mfd, memd, return_debug=True)
    assert all(torch.equal(a, b) for a, b in zip(mask, mask2)) and all(torch.equal(a, b) for a, b in zip(emb, emb2))
    cls1, emb1, mask1, dbg1 = head.decoder_forward(mfd[:1].contiguous(), [m[:1].contiguous() for m in memd],
                                                   return_debug=True)
    for j in range(10):
        assert torch.equal(mask1[j][0], mask[j][0]) and torch.equal(emb1[j][0], emb[j][0])
    # first head call only depends on query_feat: compare with the oracle at full size
    ref0 = O.head_call(sd, sd['query_feat.weight'][None], mf[:1], sizes[0])
    assert float((mask[0][0].cpu() - ref0[2][0]).abs().max()) < 5e-4
    assert np.array_equal(_bits_np(dbg['bitmaps'][0][:1]), O.pack_mask_bits(ref0[3]).numpy())


# -------------------------------------------------------------------- grounding side
@pytest.mark.parametrize('name', list(cases.GROUNDING_CASES))
def test_grounding_loss_matches_reference_golden(name):
    gold = np.load(os.path.join(GOLD, 'grounding.npz'))
    pred, cap, m = cases.grounding_tensors(name)
    sd = synth.make_params(seed=1, num_queries=pred.shape[1])
    head = _head(sd, pred.shape[1])
    loss = head.grounding_loss(pred.to(DEV), cap.to(DEV), m.to(DEV), loss_weight=2.0)
    want = float(gold[name + '_loss'])
    assert abs(float(loss) - want) < 1e-4 * max(1.0, abs(want)), (float(loss), want)
    assert abs(float(loss) - float(O.grounding_loss(pred, cap, m, 10.0, 2.0))) < 1e-4 * max(1.0, abs(want))


@pytest.mark.parametrize('name', list(cases.GROUNDING_CASES) + ['b6_d100'])
def test_grounding_loss_gradient_matches_reference_golden(name):
    """d loss / d cls_emb_pred from cgg_grounding_loss_backward against the gradients the unmodified reference
    produced (tests/golden/make_golden.py: strided sample + abs-sum) and the oracle's autograd.  b6_d100 is case b6
    cut to D = 100: not a multiple of 64, so loss and gradient take the SIMT route instead of the tcgen05 GEMMs;
    there is no golden file for that width, so it is checked against the oracle only (loss included)."""
    from cgg_b200.grounding import GroundingLossB200
    gold = np.load(os.path.join(GOLD, 'grounding.npz'))
    pred, cap, m = cases.grounding_tensors(name.replace('_d100', ''))
    if name.endswith('_d100'):
        pred, cap = pred[..., :100].contiguous(), cap[..., :100].contiguous()
    p_dev = pred.to(DEV).requires_grad_(True)
    loss = GroundingLossB200(loss_weight=2.0)(p_dev, cap.to(DEV), m.to(DEV), 10.0)
    (loss * 1.0).backward()
    g = p_dev.grad.cpu()
    p_ref = pred.clone().requires_grad_(True)
    ref_loss = O.grounding_loss(p_ref, cap, m, 10.0, 2.0)
    ref_loss.backward()
    assert abs(float(loss) - float(ref_loss)) < 1e-4 * max(1.0, abs(float(ref_loss)))
    scale = float(p_ref.grad.abs().max())
    assert float((g - p_ref.grad).abs().max()) <= 2e-5 * scale
    if name in cases.GROUNDING_CASES:
        want = gold[name + '_grad_sample']
        np.testing.assert_allclose(g.flatten()[::cases.GRAD_SAMPLE_STRIDE].numpy(), want, atol=2e-5 * scale, rtol=0)
        abssum = float(gold[name + '_grad_abssum'])
        assert abs(float(g.double().abs().sum()) - abssum) <= 1e-4 * abssum
    # upstream scaling goes through
    p2 = pred.to(DEV).requires_grad_(True)
    (GroundingLossB200(loss_weight=2.0)(p2, cap.to(DEV), m.to(DEV), 10.0) * 0.25).backward()
    torch.testing.assert_close(p2.grad, p_dev.grad * 0.25, rtol=1e-6, atol=0)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_pred_emb_norm(precision):
    """head.py:743-744: unit-norm embedding predictions, both modes, against the oracle."""
    Q, B = 32, 2
    sd = synth.make_params(seed=12, num_queries=Q, perturb=True)
    mf, mems = synth.make_inputs(12, B, 256, 256)
    if precision == 'bf16':
        mf, mems = mf.bfloat16().float(), [m.bfloat16().float() for m in mems]
    ref = O.decoder_forward(sd, mf, mems, pred_emb_norm=True)
    head = build_head_from_state_dict(sd, Q, 49, precision, DEV, pred_emb_norm=True)
    dt = torch.float32 if precision == 'fp32' else torch.bfloat16
    cls, emb, mask = head.decoder_forward(mf.to(DEV).to(dt), [m.to(DEV).to(dt) for m in mems])
    for j in (0, 9):
        scale = float(ref['emb'][j].abs().max())
        # fp32: absolute; bf16: relative to the largest component (free-running at j = 9, hence the wider band)
        tol = 2e-5 if precision == 'fp32' else (1e-2 if j == 0 else 5e-2) * scale
        assert float((emb[j].cpu() - ref['emb'][j]).abs().max()) <= tol
        assert float((emb[j].norm(dim=-1) - 1).abs().max()) < 1e-5


def test_class_embedding_logits_are_differentiable():
    """`_get_cls_emb_logits` (head.py:631-648) through cgg_similarity: value and both gradients vs torch."""
    from cgg_b200.grounding import similarity
    g = torch.Generator().manual_seed(3)
    a = torch.randn((200, 768), generator=g)
    b = torch.randn((49, 768), generator=g)
    w = torch.randn((200, 49), generator=g)
    a_ref, b_ref = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ((a_ref @ b_ref.t()) * 0.1 * w).sum().backward()
    a_d, b_d = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
    out = similarity(a_d, b_d, 0.1)
    (out * w.to(DEV)).sum().backward()
    torch.testing.assert_close(out.detach().cpu(), (a @ b.t()) * 0.1, rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(a_d.grad.cpu(), a_ref.grad, rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(b_d.grad.cpu(), b_ref.grad, rtol=1e-5, atol=1e-4)


def test_embedding_side_matches_reference_golden():
    gold = np.load(os.path.join(GOLD, 'embeddings.npz'))
    sd = synth.make_params(seed=9, num_queries=16)
    head = _head(sd, 16)
    ids, mask, table, _, _ = synth.make_captions(5, 4, vocab=400 + 1000)
    ne = head.extract_word_embeddings(table.to(DEV), torch.from_numpy(gold['ln_w']).to(DEV),
                                      torch.from_numpy(gold['ln_b']).to(DEV), ids.to(DEV))
    np.testing.assert_allclose(ne.cpu().numpy(), gold['noun_embs'], atol=3e-5, rtol=0)
    pred = torch.from_numpy(gold['pred']).to(DEV)
    np.testing.assert_allclose(head._get_cls_emb_logits(pred).cpu().numpy(), gold['logits'], atol=3e-4, rtol=0)
    np.testing.assert_allclose(head.test_time_att(pred, ne[0]).cpu().numpy(), gold['att'], atol=3e-4, rtol=0)


def _free_run_vs_oracle(sd, mf, mems, head, bit_bar, mask_tol, emb_tol):
    """All 10 head calls of a free-running forward against the oracle on the same inputs.  Free-running, one
    attention-mask bit that sits on the threshold (|logit| < 1e-5, the teacher-forced test shows these are the only
    disagreements) may flip under a different fp32 summation order and moves that query's later outputs by ~1e-3 of
    the range; hence 5e-3 here against 2e-4..5e-4 teacher-forced."""
    ref = O.decoder_forward(sd, mf, mems)
    cls, emb, mask, dbg = head.decoder_forward(mf.to(DEV), [m.to(DEV) for m in mems], return_debug=True)
    for j in range(10):
        rng = float(ref['mask'][j].abs().max())
        assert float((mask[j].cpu() - ref['mask'][j]).abs().max()) < mask_tol * rng, 'mask logits, head call %d' % j
        assert float((emb[j].cpu() - ref['emb'][j]).abs().max()) < emb_tol * float(ref['emb'][j].abs().max()), j
        assert float((cls[j].cpu() - ref['cls'][j]).abs().max()) < emb_tol * float(ref['cls'][j].abs().max()), j
        if j < 9:
            want = O.pack_mask_bits(ref['masked'][j]).numpy()
            diff = np.bitwise_xor(_bits_np(dbg['bitmaps'][j]), want)
            agree = 1.0 - np.unpackbits(diff.view(np.uint8)).sum() / ref['masked'][j].numel()
            assert agree >= bit_bar, (j, agree)


def test_fp32_full_size_1024_all_head_calls_vs_oracle():
    """BASELINE configs[1] shape (1024x1024, Q=100): every one of the 10 head calls against the oracle, fp32 mode."""
    sd = synth.make_params(seed=0, num_queries=100)
    mf, mems = synth.make_inputs(0, 1, 1024, 1024)
    _free_run_vs_oracle(sd, mf, mems, _head(sd, 100), bit_bar=0.9999, mask_tol=5e-3, emb_tol=5e-3)


def test_fp32_demo_shape_1056x800_all_head_calls_vs_oracle():
    """BASELINE configs[0] shape: the notebook demo's 1056x800 padded input (ragged key counts 825 / 3300 / 13200,
    W/4 = 200), fp32 mode, all head calls."""
    sd = synth.make_params(seed=3, num_queries=100, perturb=True)
    mf, mems = synth.make_inputs(2, 1, 1056, 800)
    _free_run_vs_oracle(sd, mf, mems, _head(sd, 100), bit_bar=0.9999, mask_tol=5e-3, emb_tol=5e-3)


def test_fp32_osps_q200_ncls118_vs_oracle():
    """BASELINE configs[3] head shape: 200 queries, 118 class rows, real class embeddings, at 512x512."""
    c = dict(cases.HEAD_CASES['osps_q200'], height=512, width=512, batch=2)
    sd, mf, mems = cases.case_tensors(c)
    _free_run_vs_oracle(sd, mf, mems, _head(sd, 200), bit_bar=0.9999, mask_tol=5e-3, emb_tol=5e-3)
