"""GPU tests of the fused panoptic output (`cgg_panoptic_fuse`, postprocess.panoptic_postprocess_fused /
fusion_simple_test) against the plain-torch oracle (oracle/panoptic_oracle.py: mmdet 2.28.2
MaskFormerFusionHead.panoptic_postprocess on the class-embedding probabilities) applied to the same low-resolution
logits.  Random-init heads keep no query (no class probability passes 0.8), so every case plants its kept queries."""
import pytest
import torch

from cgg_b200 import lib as L
from cgg_b200 import postprocess as P
from cgg_b200 import synth
from cgg_b200.head import build_head_from_state_dict
from oracle import panoptic_oracle as PO

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _head(Q, ncls1, num_stuff, precision='fp32', seed=3):
    sd = synth.make_params(seed=seed, num_queries=Q, num_classes_p1=ncls1)
    return build_head_from_state_dict(sd, Q, ncls1, precision, DEV, num_stuff_classes=num_stuff)


def _planted_probs(g, Q, C, frac_kept):
    """(Q, C+1): a fraction of the queries kept (distinct scores in (0.82, 0.99), random labels), the others void winners
    or below the threshold."""
    probs = torch.full((Q, C + 1), 0.0)
    r = torch.rand(Q, generator=g)
    labels = torch.randint(0, C, (Q,), generator=g)
    scores = 0.82 + 0.17 * torch.randperm(Q, generator=g).float() / Q
    for q in range(Q):
        if r[q] < frac_kept:
            lab, sc = int(labels[q]), float(scores[q])
        elif r[q] < (1 + frac_kept) / 2:
            lab, sc = C, 0.9
        else:
            lab, sc = int(labels[q]), 0.4
        probs[q] = (1.0 - sc) / C
        probs[q, lab] = sc
    return probs


def _blobs(g, Q, h, w):
    yy = torch.arange(h, dtype=torch.float32)[:, None]
    xx = torch.arange(w, dtype=torch.float32)[None, :]
    c = torch.rand((Q, 3), generator=g)
    cy, cx, r = c[:, 0, None, None] * h, c[:, 1, None, None] * w, 2.0 + c[:, 2, None, None] * h / 5
    d2 = (yy - cy) ** 2 + (xx - cx) ** 2
    return 6.0 * (1.0 - d2 / r ** 2) + 0.5 * torch.randn((Q, h, w), generator=g)


METAS = [dict(batch_input_shape=(256, 320), img_shape=(250, 300, 3), ori_shape=(375, 450, 3)),
         dict(batch_input_shape=(256, 320), img_shape=(256, 277, 3), ori_shape=(511, 553, 3))]


def _near_ties(prob_masks):
    """pixels whose top-two score * sigmoid differ by at most 4 fp32 ulps of the larger"""
    if prob_masks.shape[0] < 2:
        return torch.zeros(prob_masks.shape[-2:], dtype=torch.bool, device=prob_masks.device)
    top = prob_masks.topk(2, dim=0).values
    return (top[0] - top[1]) <= 4 * torch.finfo(torch.float32).eps * top[0]


def _compare(pan, stats, b, want, want_st, exact=False):
    near = _near_ties(want_st['prob_masks'])
    mism = pan.cpu() != want.cpu()
    near = near.cpu()
    assert not (mism & ~near).any(), int((mism & ~near).sum())
    assert int(mism.sum()) <= 1e-5 * mism.numel()
    if exact or not near.any():
        assert not mism.any()
        for k in ('mask_area', 'original_area', 'seg_value'):
            assert torch.equal(stats[k][b].cpu().long(), want_st[k]), k
    return int(near.sum())


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('rescale', [False, True])
@pytest.mark.parametrize('Q,ncls1,nstuff', [(100, 49, 8), (200, 118, 53)])
@pytest.mark.parametrize('filter_low_score', [False, True])
def test_kernel_matches_oracle(dtype, rescale, Q, ncls1, nstuff, filter_low_score):
    head = _head(Q, ncls1, nstuff)
    C = ncls1 - 1
    g = torch.Generator().manual_seed(Q + 7 * int(rescale) + 3 * int(filter_low_score))
    probs = torch.stack([_planted_probs(g, Q, C, 0.3) for _ in range(2)]).to(DEV)
    logits = torch.stack([_blobs(g, Q, 64, 80) for _ in range(2)]).to(DEV).to(dtype)
    cfg = dict(object_mask_thr=0.8, iou_thr=0.8, filter_low_score=filter_low_score)
    maps, st = P.panoptic_postprocess_fused(head, probs, logits, METAS, rescale=rescale, test_cfg=cfg, stats=True)
    segs = 0
    for b in range(2):
        want, want_st = PO.panoptic_from_lowres(probs[b], logits[b].float(), METAS[b], head.num_things_classes, rescale,
                                                **cfg)
        assert maps[b].shape == want.shape and maps[b].dtype == torch.int32
        assert maps[b].untyped_storage().data_ptr() == maps[0].untyped_storage().data_ptr()   # views of one buffer
        _compare(maps[b], st, b, want, want_st)
        segs += int((want_st['seg_value'] >= 0).sum())
        assert int(want_st['keep'].sum()) >= 10
    assert segs >= 3                                                   # the planted cases do produce segments


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('frac', [0.0, 1.0])
def test_zero_kept_and_all_kept(dtype, frac):
    Q, ncls1 = 100, 49
    head = _head(Q, ncls1, 8)
    g = torch.Generator().manual_seed(11)
    probs = torch.stack([_planted_probs(g, Q, ncls1 - 1, frac) for _ in range(2)]).to(DEV)
    logits = torch.stack([_blobs(g, Q, 64, 80) for _ in range(2)]).to(DEV).to(dtype)
    maps, st = P.panoptic_postprocess_fused(head, probs, logits, METAS, rescale=True, stats=True)
    for b in range(2):
        want, want_st = PO.panoptic_from_lowres(probs[b], logits[b].float(), METAS[b], head.num_things_classes, True)
        assert int(want_st['keep'].sum()) == (0 if frac == 0 else Q)
        _compare(maps[b], st, b, want, want_st)
        if frac == 0:
            assert (maps[b] == ncls1 - 1).all()


def _identity_meta(h, w):
    return dict(batch_input_shape=(h, w), img_shape=(h, w, 3), ori_shape=(h, w, 3))


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_sigmoid_cutoff(dtype):
    """Logits at and around the sigmoid >= 0.5 cutoff, with an identity resample (batch_input_shape = the logits' size)
    so that the kernel sees exactly these values: the flag, original_area and the filter_low_score map are exact."""
    Q, ncls1, h, w = 4, 49, 40, 64
    head = _head(Q, ncls1, 8)
    ticks = torch.tensor([0.0, -0.0, 1e-8, -1e-8, -3e-8, -6e-8, -6.5e-8, -1e-7, -1.5e-7, -1.7881391e-07, -1.7881392e-07,
                          -2e-7, -3e-7, 1e-7, -1e-6, 1e-6])     # sigma < 0.5  <=>  x <= -1.7881392e-07 (DESIGN §2)
    base = ticks.repeat(h * w // ticks.numel() + 1)[:h * w].view(h, w)
    if dtype == torch.bfloat16:
        base = base.to(torch.bfloat16).float()
    logits = torch.stack([base, base.flip(1) * 3, -base, torch.full((h, w), -20.0)])[None]
    probs = torch.stack([torch.tensor([0.9 if c == 3 else 0.1 / 48 for c in range(49)]),
                         torch.tensor([0.85 if c == 40 else 0.15 / 48 for c in range(49)]),
                         torch.tensor([0.95 if c == 5 else 0.05 / 48 for c in range(49)]),
                         torch.tensor([0.99 if c == 7 else 0.01 / 48 for c in range(49)])])[None]
    meta = [_identity_meta(h, w)]
    for flt in (False, True):
        cfg = dict(object_mask_thr=0.8, iou_thr=0.0, filter_low_score=flt)
        maps, st = P.panoptic_postprocess_fused(head, probs.to(DEV), logits.to(DEV).to(dtype), meta, test_cfg=cfg,
                                                stats=True)
        # the oracle on the GPU: torch's CUDA sigmoid is the one whose cutoff the kernel reproduces
        want, want_st = PO.panoptic_from_lowres(probs[0].to(DEV), logits[0].to(DEV).to(dtype).float(), meta[0],
                                                head.num_things_classes, **cfg)
        _compare(maps[0], st, 0, want, want_st, exact=True)
        assert 0 < int(want_st['original_area'][0]) < h * w


HAND = [  # (spec [(label, score)], strips [(a, b)], filter_low_score) -- the known-answer cases of test_panoptic_cpu.py
    ([(2, 0.9), (4, 0.95)], [(0, 100), (79, 200)], False),            # ratio 0.79: dropped
    ([(2, 0.9), (4, 0.95)], [(0, 100), (80, 200)], False),            # ratio 0.80: kept
    ([(3, 0.9)], [(0, 100)], False),                                  # mask_area 200 > filtered 100
    ([(3, 0.9)], [(0, 100)], True),
    ([(7, 0.9), (1, 0.9), (7, 0.9)], [(0, 60), (60, 120), (120, 200)], False),   # stuff merge
    ([(0, 0.9), (1, 0.85), (2, 0.95), (5, 0.9)], [(0, 50), (50, 100), (60, 150), (150, 200)], False),  # ids skip
    ([(10, 0.9), (4, 0.9), (5, 0.9)], [(0, 0), (0, 200), (0, 200)], False),     # exact tie -> lower kept index
]


@pytest.mark.parametrize('case', range(len(HAND)))
def test_known_answer_cases(case):
    spec, strips, flt = HAND[case]
    C, Q = 10, len(spec)
    head = _head(Q, C + 1, 4)                                          # things 0..5, stuff 6..9
    probs = torch.empty((Q, C + 1))
    for q, (lab, sc) in enumerate(spec):
        probs[q] = (1.0 - sc) / C
        probs[q, lab] = sc
    logits = torch.full((Q, 4, 200), -5.0)
    for q, (a, b) in enumerate(strips):
        logits[q, :, a:b] = 5.0
    meta = [_identity_meta(4, 200)]
    cfg = dict(filter_low_score=flt)
    maps, st = P.panoptic_postprocess_fused(head, probs[None].to(DEV), logits[None].to(DEV), meta, test_cfg=cfg, stats=True)
    want, want_st = PO.panoptic_from_lowres(probs.to(DEV), logits.to(DEV), meta[0], head.num_things_classes, **cfg)
    _compare(maps[0], st, 0, want, want_st, exact=True)


def _plant(head, emb, g, frac=0.3):
    """cls_emb rows of a fraction of the queries set to a scaled class_embs row: softmax(emb @ class_embs^T) then peaks
    at that class with a probability above 0.8."""
    B, Q, _ = emb.shape
    ce = head.class_embs.float()
    C = ce.shape[0] - 1
    for b in range(B):
        for q in range(Q):
            if float(torch.rand((), generator=g)) < frac:
                lab = int(torch.randint(0, C, (), generator=g))
                emb[b, q] = ce[lab] * (6.0 + 4.0 * float(torch.rand((), generator=g))) / ce[lab].norm() ** 2
    return emb


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_fusion_simple_test_end_to_end(precision):
    Q, ncls1, B = 100, 49, 2
    head = _head(Q, ncls1, 8, precision, seed=5)
    head.test_cfg = dict(panoptic_on=True, instance_on=True, max_per_image=100)
    mf, mems = synth.make_inputs(8, B, 256, 320)
    with torch.no_grad():
        cls, emb, masks = head.decoder_forward(mf.to(DEV), [m.to(DEV) for m in mems])
    g = torch.Generator().manual_seed(1)
    e = _plant(head, emb[-1].clone(), g)
    lowres = masks[-1]
    assert lowres.dtype == (torch.bfloat16 if precision == 'bf16' else torch.float32)
    res = P.fusion_simple_test(head, cls[-1], e, lowres, METAS, rescale=True)
    probs = P.class_probs(head, cls[-1], e)
    torch.testing.assert_close(probs, torch.softmax(e @ head.class_embs.float().t(), -1), rtol=0, atol=1e-4)
    ins = P.instance_postprocess_emb_fused(head, e, lowres, head.class_embs, METAS, rescale=True)
    kept = 0
    for b in range(B):
        want, want_st = PO.panoptic_from_lowres(probs[b], lowres[b].float(), METAS[b], head.num_things_classes, True)
        kept += int(want_st['keep'].sum())
        near = _near_ties(want_st['prob_masks']).cpu()
        mism = res[b]['pan_results'].cpu() != want.cpu()
        assert not (mism & ~near).any() and int(mism.sum()) <= 1e-5 * mism.numel()
        (l0, b0, m0, s0), (l1, b1, m1, s1) = res[b]['ins_results'], ins[b]
        assert torch.equal(l0, l1) and torch.equal(m0, m1) and torch.equal(b0[:, :4], b1[:, :4]) and s0 == s1
        # the sigmoid sums behind the detection scores are float atomics: equal up to summation order
        torch.testing.assert_close(b0[:, 4], b1[:, 4], rtol=1e-5, atol=1e-7)
    assert kept >= 20


def test_semantic_on_raises():
    head = _head(8, 49, 8)
    head.test_cfg = dict(semantic_on=True)
    x = torch.zeros((1, 8, 4, 4), device=DEV)
    with pytest.raises(NotImplementedError):
        P.fusion_simple_test(head, torch.zeros((1, 8, 49), device=DEV), torch.zeros((1, 8, 768), device=DEV), x,
                             [_identity_meta(4, 4)])


def _case(Q=100, ncls1=49, seed=21):
    head = _head(Q, ncls1, 8)
    g = torch.Generator().manual_seed(seed)
    probs = torch.stack([_planted_probs(g, Q, ncls1 - 1, 0.3) for _ in range(2)]).to(DEV)
    logits = torch.stack([_blobs(g, Q, 64, 80) for _ in range(2)]).to(DEV).to(torch.bfloat16)
    return head, probs, logits, g


def test_no_host_sync():
    head, probs, logits, _ = _case()
    metas = [dict(batch_input_shape=(256, 320), img_shape=(241, 307, 3), ori_shape=(300, 400, 3)),
             dict(batch_input_shape=(256, 320), img_shape=(199, 320, 3), ori_shape=(250, 390, 3))]
    P.cls_emb_scores(head, torch.zeros((1, 1, 768), device=DEV), head.class_embs)       # runtime created outside
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        maps = P.panoptic_postprocess_fused(head, probs, logits, metas, rescale=True)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    want, _ = PO.panoptic_from_lowres(probs[1], logits[1].float(), metas[1], head.num_things_classes, True)
    assert maps[1].shape == want.shape


def test_cuda_graph_replay_matches_eager():
    head, probs, logits, g = _case(seed=23)
    static_logits, static_probs = logits.clone(), probs.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        P.panoptic_postprocess_fused(head, static_probs, static_logits, METAS, rescale=True)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with L.no_gc_during_capture(), torch.cuda.graph(graph):
        maps = P.panoptic_postprocess_fused(head, static_probs, static_logits, METAS, rescale=True)
    graph.replay()
    eager = P.panoptic_postprocess_fused(head, probs, logits, METAS, rescale=True)
    for a, b in zip(maps, eager):
        assert torch.equal(a, b)
    new_logits = torch.stack([_blobs(g, 100, 64, 80) for _ in range(2)]).to(DEV).to(torch.bfloat16)
    static_logits.copy_(new_logits)
    graph.replay()
    eager = P.panoptic_postprocess_fused(head, probs, new_logits, METAS, rescale=True)
    for a, b in zip(maps, eager):
        assert torch.equal(a, b)
    first = P.panoptic_postprocess_fused(head, probs, logits, METAS, rescale=True)
    assert any(not torch.equal(a, b) for a, b in zip(first, eager))   # the replay did see the new logits
