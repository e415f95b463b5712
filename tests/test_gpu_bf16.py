"""GPU parity tests of the throughput mode (CGG_BF16: bf16 operands on tcgen05, fp32 accumulate)
against the oracle's fp32 results.  Tolerances are the ones BASELINE.json states for bf16 mode:
  * mask / class / grounding logits: max-abs error <= 1e-2 of the logit range,
  * attention-mask bits: >= 99.9 % agreement,
  * final mask IoU >= 0.99,
all against the reference-equivalent fp32 path on identical inputs and weights."""
import numpy as np
import pytest
import torch

from oracle import cgg_oracle as O
from cgg_b200 import synth
from cgg_b200.head import build_head_from_state_dict

pytestmark = pytest.mark.gpu
DEV = 'cuda'
REL_TOL = 1e-2
BIT_AGREE = 0.999
IOU_MIN = 0.99


def _unpack(bm, K):
    w = bm.cpu().numpy().astype(np.int32)
    bits = np.unpackbits(w.view(np.uint8), bitorder='little').reshape(w.shape[0], w.shape[1], -1)[:, :, :K]
    return torch.from_numpy(bits.astype(bool))


def _rel(got, want):
    return float((got.float().cpu() - want).abs().max()) / float(want.abs().max())


def _setup(Q, B, H, W, pseed, iseed):
    sd = synth.make_params(seed=pseed, num_queries=Q, perturb=True)
    mf, mems = synth.make_inputs(iseed, B, H, W)
    # the bf16 path consumes bf16 pixel-decoder outputs; the oracle sees the SAME (rounded) values
    mf, mems = mf.bfloat16().float(), [m.bfloat16().float() for m in mems]
    head = build_head_from_state_dict(sd, Q, 49, 'bf16', DEV)
    return sd, mf, mems, head


# 352x288 and 1056x800 have key counts that are not multiples of 8 (11x9, 22x18; 33x25, 66x50 = the reference demo's
# 1056x800): those levels are re-pitched for TMA inside cgg_kv_project.  Odd tile counts (256x256: the 8x8 level is one
# 128-key tile; 352x288) leave the second CTA of the last pair wholly past the end.  Q = 128 and 240 take the pixel-on-lane
# pair einsum (one and two N tiles per head call), Q = 300 also two attention-mask query slices.
@pytest.mark.parametrize('Q,B,H,W', [(100, 2, 256, 256), (37, 1, 256, 320), (200, 1, 256, 256), (300, 1, 256, 256),
                                     (100, 2, 352, 288), (100, 1, 1056, 800), (128, 1, 256, 256), (240, 1, 256, 256)])
def test_bf16_teacher_forced_layers(Q, B, H, W):
    sd, mf, mems, head = _setup(Q, B, H, W, 31, 7)
    ref = O.decoder_forward(sd, mf, mems)
    dev = torch.device(DEV, 0)
    rt = head._runtime(dev)
    sizes = [tuple(m.shape[-2:]) for m in mems]
    rt.prepare(mf.shape[2], mf.shape[3], sizes, B)
    mfd = mf.to(dev).bfloat16()
    rt.kv_project([m.to(dev).bfloat16() for m in mems])
    for i in range(9):
        x = ref['x'][i].to(dev).contiguous()
        cls, emb, mask, me, bm, am = rt.head_call(x, mfd, i % 3)
        assert _rel(cls, ref['cls'][i]) < REL_TOL and _rel(emb, ref['emb'][i]) < REL_TOL
        assert _rel(mask, ref['mask'][i]) < REL_TOL, 'mask logits, head call %d' % i
        K = sizes[i % 3][0] * sizes[i % 3][1]
        agree = float((_unpack(bm, K) == ref['masked'][i]).float().mean())
        assert agree >= BIT_AGREE, 'attention-mask bit agreement %.5f at head call %d' % (agree, i)
        want_bits = O.pack_mask_bits(ref['masked'][i]).to(dev)
        x_out = rt.decoder_layer(i, x, want_bits, ref['masked'][i].all(-1).to(torch.uint8).to(dev))
        assert _rel(x_out, ref['x'][i + 1]) < REL_TOL, 'decoder layer %d' % i


def _iou(got, want):
    inter = (got & want).flatten(2).sum(-1).float()
    union = (got | want).flatten(2).sum(-1).float().clamp(min=1)
    return float((inter / union).mean())


def _free_running(Q, B, H, W, pseed, iseed, ncls1=49, class_embs=None):
    """Free-running forward, ALL 10 head calls, at the BASELINE tolerances (no loosened bars): max-abs <= 1e-2 of the
    logit range for mask / class / embedding logits, >= 99.9 % attention-mask bits on every head call, final-mask
    IoU >= 0.99."""
    sd = synth.make_params(seed=pseed, num_queries=Q, perturb=True, num_classes_p1=ncls1)
    if class_embs is not None:
        sd['class_embs'] = class_embs
    mf, mems = synth.make_inputs(iseed, B, H, W)
    mf, mems = mf.bfloat16().float(), [m.bfloat16().float() for m in mems]
    head = build_head_from_state_dict(sd, Q, ncls1, 'bf16', DEV)
    ref = O.decoder_forward(sd, mf, mems)
    cls, emb, mask, dbg = head.decoder_forward(mf.to(DEV).bfloat16(), [m.to(DEV).bfloat16() for m in mems],
                                               return_debug=True)
    assert mask[0].dtype == torch.bfloat16 and len(mask) == 10
    sizes = [tuple(m.shape[-2:]) for m in mems]
    for j in range(10):
        assert _rel(mask[j], ref['mask'][j]) <= REL_TOL, ('mask', j, _rel(mask[j], ref['mask'][j]))
        assert _rel(emb[j], ref['emb'][j]) <= REL_TOL, ('emb', j, _rel(emb[j], ref['emb'][j]))
        assert _rel(cls[j], ref['cls'][j]) <= REL_TOL, ('cls', j, _rel(cls[j], ref['cls'][j]))
        if j < 9:
            K = sizes[j % 3][0] * sizes[j % 3][1]
            agree = float((_unpack(dbg['bitmaps'][j], K) == ref['masked'][j]).float().mean())
            assert agree >= BIT_AGREE, (j, agree)
    assert _iou(mask[9].float().cpu() > 0, ref['mask'][9] > 0) >= IOU_MIN
    # grounding / class-embedding logits from the final embeddings (head.py:631-648)
    logits = head._get_cls_emb_logits(emb[9])
    want_l = O.cls_emb_logits(ref['emb'][9], sd['class_embs'], 10.0)
    assert _rel(logits, want_l) <= REL_TOL


def test_bf16_free_running_1024_all_head_calls():
    """BASELINE configs[1] shape: 1024x1024, Q=100, B=2."""
    _free_running(100, 2, 1024, 1024, 33, 9)


def test_bf16_free_running_768():
    _free_running(100, 2, 768, 768, 5, 3)


def test_bf16_free_running_osps_q200_ncls118():
    """BASELINE configs[3] head shape: 200 queries, 118 class rows, the reference's real class embeddings."""
    import cases
    _free_running(200, 2, 512, 512, 8, 5, ncls1=118, class_embs=cases.real_class_embs('coco_panoptic_p20'))


@pytest.mark.parametrize('H,W,pseed,iseed', [(256, 256, 33, 9), (512, 512, 5, 3)])
def test_bf16_free_running_few_keys_reported(H, W, pseed, iseed):
    """Small inputs: at 256x256 (512x512) the 1/32 level has 64 (256) keys, so ONE flipped attention-mask bit moves a
    query's softmax by ~1/32 (1/128) and the free-running max-abs error is set by such discrete events rather than by
    rounding (CPU study tools/bf16_drift_study.py, DESIGN.md section 3: K/V stored in bf16 alone gives 1.3e-2 ..
    2.1e-2 at 256x256 and 6e-4 at 1024x1024; measured on the GPU at 512x512: 1.3e-2 on one embedding logit).  The stated
    tolerances are asserted teacher-forced on these shapes (test above) and free-running from 768x768 up (the metric is
    quoted at 1024x1024); here the IoU and bit bars are asserted and the float errors are printed."""
    Q, B = 100, 2
    sd, mf, mems, head = _setup(Q, B, H, W, pseed, iseed)
    ref = O.decoder_forward(sd, mf, mems)
    cls, emb, mask, dbg = head.decoder_forward(mf.to(DEV).bfloat16(), [m.to(DEV).bfloat16() for m in mems],
                                               return_debug=True)
    sizes = [tuple(m.shape[-2:]) for m in mems]
    for j in range(9):
        K = sizes[j % 3][0] * sizes[j % 3][1]
        agree = float((_unpack(dbg['bitmaps'][j], K) == ref['masked'][j]).float().mean())
        assert agree >= BIT_AGREE, (j, agree)
    assert _iou(mask[9].float().cpu() > 0, ref['mask'][9] > 0) >= IOU_MIN
    print('%dx%d free-running: mask %.3g emb %.3g of range' % (H, W, _rel(mask[9], ref['mask'][9]), _rel(emb[9], ref['emb'][9])))
    assert _rel(mask[9], ref['mask'][9]) < 3 * REL_TOL and _rel(emb[9], ref['emb'][9]) < 3 * REL_TOL


def test_bf16_cuda_graph_matches_eager_and_survives_reprepare():
    """cuda_graph=True (the path bench.py measures): replay == eager bit for bit; A -> B -> A shape changes and a
    weight update between replays must re-capture instead of replaying a graph that points at freed tables."""
    Q = 100
    sd = synth.make_params(seed=21, num_queries=Q, perturb=True)
    eager = build_head_from_state_dict(sd, Q, 49, 'bf16', DEV)
    graph = build_head_from_state_dict(sd, Q, 49, 'bf16', DEV, cuda_graph=True)

    def inputs(iseed, B, H, W):
        mf, mems = synth.make_inputs(iseed, B, H, W)
        return mf.to(DEV).bfloat16(), [m.to(DEV).bfloat16() for m in mems]

    def same(a, b):
        return all(torch.equal(x, y) for la, lb in zip(a, b) for x, y in zip(la, lb))

    inA, inB = inputs(1, 2, 256, 256), inputs(2, 1, 256, 320)
    for inp in (inA, inB, inA, inA):          # A -> B -> A -> A (replay)
        want = eager.decoder_forward(*inp)
        got = graph.decoder_forward(*inp)
        torch.cuda.synchronize()
        assert same(want, got)
    # fresh tensors of the same shape (a real pixel decoder returns new tensors every step): no stale pointers
    inA2 = tuple(inputs(3, 2, 256, 256))
    assert same(eager.decoder_forward(*inA2), graph.decoder_forward(*inA2))
    inA3 = tuple(inputs(4, 2, 256, 256))
    assert same(eager.decoder_forward(*inA3), graph.decoder_forward(*inA3))
    # weight update between replays
    with torch.no_grad():
        for h in (eager, graph):
            h.transformer_decoder.layers[3].ffns[0].layers[1].weight.mul_(1.5)
            h.query_feat.weight.add_(0.25)
    assert same(eager.decoder_forward(*inA3), graph.decoder_forward(*inA3))


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_use_class_emb_false_returns_cls_as_emb(precision):
    """head.py:739-744 with use_class_emb=False (the class-agnostic pre-training configs, which also set
    pred_emb_norm=True): cls_emb_pred IS cls_pred, no v2l_transform, no normalisation."""
    Q, B = 32, 2
    sd = synth.make_params(seed=14, num_queries=Q, perturb=True)
    mf, mems = synth.make_inputs(6, B, 256, 256)
    mf, mems = mf.bfloat16().float(), [m.bfloat16().float() for m in mems]
    ref = O.decoder_forward(sd, mf, mems)
    sd2 = {k: v for k, v in sd.items() if not k.startswith('v2l_transform') and k != 'class_embs'}
    head = build_head_from_state_dict(sd2, Q, 49, precision, DEV, pred_emb_norm=True)
    dt = torch.float32 if precision == 'fp32' else torch.bfloat16
    cls, emb, mask = head.decoder_forward(mf.to(DEV).to(dt), [m.to(DEV).to(dt) for m in mems])
    assert all(e is c_ for e, c_ in zip(emb, cls))
    assert _rel(cls[0], ref['cls'][0]) < (1e-4 if precision == 'fp32' else REL_TOL)
    assert _rel(mask[0], ref['mask'][0]) < (1e-4 if precision == 'fp32' else REL_TOL)


def test_bf16_final_mask_only_matches_full_forward():
    """Opt-in inference shortcut: same class / embedding outputs and the same final mask, bit for bit; the nine
    intermediate masks are not produced."""
    Q, B, H, W = 100, 2, 256, 256
    sd, mf, mems, head = _setup(Q, B, H, W, 35, 11)
    mfd, memd = mf.to(DEV).bfloat16(), [m.to(DEV).bfloat16() for m in mems]
    cls, emb, mask = head.decoder_forward(mfd, memd)
    fast = build_head_from_state_dict(sd, Q, 49, 'bf16', DEV, final_mask_only=True)
    cls2, emb2, mask2 = fast.decoder_forward(mfd, memd)
    assert all(m is None for m in mask2[:-1]) and len(mask2) == 10
    assert torch.equal(mask2[-1], mask[-1])
    for a, b in zip(cls + emb, cls2 + emb2):
        assert torch.equal(a, b)


def _batched_einsum_check(Q, H, W):
    B = 2
    sd, mf, mems, head = _setup(Q, B, H, W, 35, 11)
    mfd, memd = mf.to(DEV).bfloat16(), [m.to(DEV).bfloat16() for m in mems]
    cls, emb, mask, dbg = head.decoder_forward(mfd, memd, return_debug=True)
    rt = head._runtime(torch.device(DEV, 0))
    for j in (0, 3, 9):
        _, _, m1, _, _, _ = rt.head_call(dbg['x'][j].contiguous(), mfd, j % 3, want_bits=False)
        assert torch.equal(m1, mask[j]), j
    # head calls 1..3 of the forward still have their mask embeddings in the workspace (head_call writes call slot 0):
    # one batched call over an odd number of head calls that does not start at call 0
    odd = torch.empty((3,) + tuple(mask[0].shape), dtype=torch.bfloat16, device=DEV)
    rt.mask_einsum(mfd, odd, first_call=1, num_calls=3)
    torch.cuda.synchronize()
    for i in range(3):
        assert torch.equal(odd[i], mask[1 + i]), 1 + i


def test_bf16_batched_einsum_equals_per_call_einsum():
    """The all-calls-in-one-pass einsum (A tile resident) must equal the per-call stage output, as must a pass over an
    odd number of head calls."""
    _batched_einsum_check(100, 256, 256)


@pytest.mark.parametrize('Q,H,W', [(100, 352, 288), (128, 256, 256), (240, 256, 256), (300, 256, 256)])
def test_bf16_batched_einsum_equals_per_call_einsum_other_routes(Q, H, W):
    """The same with a partial last pixel tile (352x288: 88x72 = 6336 mask pixels) and on the pixel-on-lane pair einsum
    (Q = 128: one N tile per head call; Q = 240, 300: two)."""
    _batched_einsum_check(Q, H, W)


def _full_size_properties(Q):
    """1024x1024, B=2: run-to-run determinism and per-image independence of every head call's mask, embedding and
    attention-mask bitmap, and layer-0 parity with the oracle at full size."""
    B = 2
    sd = synth.make_params(seed=0, num_queries=Q)
    mf, mems = synth.make_inputs(0, B, 1024, 1024)
    mf, mems = mf.bfloat16(), [m.bfloat16() for m in mems]
    head = build_head_from_state_dict(sd, Q, 49, 'bf16', DEV)
    mfd, memd = mf.to(DEV), [m.to(DEV) for m in mems]
    cls, emb, mask, dbg = head.decoder_forward(mfd, memd, return_debug=True)
    cls2, emb2, mask2, dbg2 = head.decoder_forward(mfd, memd, return_debug=True)
    assert all(torch.equal(a, b) for a, b in zip(mask, mask2)) and all(torch.equal(a, b) for a, b in zip(emb, emb2))
    assert all(torch.equal(a, b) for a, b in zip(dbg['bitmaps'], dbg2['bitmaps']))
    assert torch.equal(dbg['all_masked'], dbg2['all_masked'])
    cls1, emb1, mask1, dbg1 = head.decoder_forward(mfd[:1].contiguous(), [m[:1].contiguous() for m in memd],
                                                   return_debug=True)
    for j in range(10):
        assert torch.equal(mask1[j][0], mask[j][0]) and torch.equal(emb1[j][0], emb[j][0]), j
        if j < 9:
            assert torch.equal(dbg1['bitmaps'][j][0], dbg['bitmaps'][j][0]), j
    ref0 = O.head_call(sd, sd['query_feat.weight'][None], mf[:1].float(), (32, 32))
    assert _rel(mask[0][:1], ref0[2]) < REL_TOL
    agree = float((_unpack(dbg['bitmaps'][0][:1], 1024) == ref0[3]).float().mean())
    assert agree >= BIT_AGREE, agree


def test_bf16_full_size_1024_properties():
    """The benchmark's query count (Q = 100: the mask einsum runs two head calls per step)."""
    _full_size_properties(100)


@pytest.mark.parametrize('Q', [200, 300])
def test_bf16_full_size_1024_properties_other_routes(Q):
    """The same on the other mask-einsum routes: Q = 200 runs one head call per step split over the CTA pair, Q = 300
    the pixel-on-lane pair kernel with two N tiles and the attention-mask GEMM with two query slices.  (An accumulator
    overlap of the attention-mask GEMM at 129..256 queries once made two runs at Q = 200 differ within the 1e-2 bar.)"""
    _full_size_properties(Q)
