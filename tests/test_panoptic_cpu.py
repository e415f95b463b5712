"""CPU tests of the panoptic oracle (oracle/panoptic_oracle.py): pinned on HuggingFace's independent
`compute_segments` (with hf_semantics=True), and hand-built cases with known answers for mmdet 2.28.2's
`MaskFormerFusionHead.panoptic_postprocess` semantics."""
import pytest
import torch

from oracle import panoptic_oracle as PO


def planted_probs(spec, num_classes):
    """spec: list of (label, score) per query -> (Q, C+1) probabilities with `label` the argmax at `score` (label =
    num_classes is the void column); the rest of the mass spread evenly."""
    C1 = num_classes + 1
    probs = torch.empty((len(spec), C1), dtype=torch.float32)
    for q, (label, score) in enumerate(spec):
        probs[q] = (1.0 - score) / (C1 - 1)
        probs[q, label] = score
    return probs


def strip(*ranges, width=200, pos=5.0, neg=-5.0):
    """(Q, 1, width) logits: query q positive on [a, b) of ranges[q]."""
    m = torch.full((len(ranges), 1, width), neg)
    for q, (a, b) in enumerate(ranges):
        m[q, 0, a:b] = pos
    return m


# ---------------------------------------------------------------- pinned on HuggingFace's compute_segments

def _seeded_case(seed, Q=16, C=20, num_things=12, H=48, W=56):
    g = torch.Generator().manual_seed(seed)
    spec = []
    for q in range(Q):
        r = float(torch.rand((), generator=g))
        label = int(torch.randint(0, num_things, (), generator=g))
        if r < 0.3:
            spec.append((C, 0.9))                                    # void winner: never kept
        elif r < 0.45:
            spec.append((label, 0.5))                                # below the threshold
        else:
            spec.append((label, 0.81 + 0.18 * float(torch.rand((), generator=g))))
    # HF reuses the fused segment's id as its running counter, so a stuff class that repeats after other segments could
    # collide with a later new id; end the query list with repeats of ONE stuff class so the two agree on the partition
    stuff = num_things + 1
    spec[-3:] = [(stuff, 0.95), (stuff, 0.9), (stuff, 0.92)]
    spec[2] = (stuff, 0.93)
    spec[5] = (num_things + 3, 0.9)
    return planted_probs(spec, C), blobs(g, Q, H // 4, W // 4)


def blobs(g, Q, h, w):
    """(Q, h, w) low-resolution logits: one noisy disc per query at a random centre and radius, so that some queries
    win most of their own disc and others lose it to an overlapping, higher-scoring one."""
    yy = torch.arange(h, dtype=torch.float32)[:, None]
    xx = torch.arange(w, dtype=torch.float32)[None, :]
    c = torch.rand((Q, 3), generator=g)
    cy, cx, r = c[:, 0, None, None] * h, c[:, 1, None, None] * w, 1.5 + c[:, 2, None, None] * h / 6
    d2 = (yy - cy) ** 2 + (xx - cx) ** 2
    return 6.0 * (1.0 - d2 / r ** 2) + 0.5 * torch.randn((Q, h, w), generator=g)


def _partition(values, void):
    """pixel values -> canonical segment index per pixel (first appearance order), void -> -1."""
    flat = values.flatten().tolist()
    ids, out = {}, []
    for v in flat:
        if v == void:
            out.append(-1)
        else:
            out.append(ids.setdefault(v, len(ids)))
    return out, ids


@pytest.mark.parametrize('seed', [0, 1, 2, 3])
def test_oracle_hf_semantics_matches_compute_segments(seed):
    from transformers.models.mask2former.image_processing_mask2former import compute_segments
    C, num_things = 20, 12
    probs, lowres = _seeded_case(seed, C=C, num_things=num_things)
    meta = dict(batch_input_shape=(48, 56), img_shape=(45, 50), ori_shape=(60, 70))
    mp = PO.resample_logits(lowres, meta['batch_input_shape'], meta['img_shape'], meta['ori_shape'])
    pan, st = PO.panoptic_postprocess(probs, mp, num_things, hf_semantics=True)
    keep = st['keep']
    assert 5 <= int(keep.sum()) < probs.shape[0]
    scores, labels = probs.max(-1)
    seg, segments = compute_segments(mp.sigmoid()[keep].clone(), scores[keep], labels[keep], 0.5, 0.8,
                                     label_ids_to_fuse=set(range(num_things, C)), target_size=None)
    assert len(segments) >= 3
    ours, our_ids = _partition(pan, C)
    theirs, their_ids = _partition(seg, 0)
    assert ours == theirs                                            # same partition of the pixels into segments
    hf_label = {s['id']: s['label_id'] for s in segments}
    for v, i in our_ids.items():                                     # and each segment's label
        hf_id = [k for k, j in their_ids.items() if j == i][0]
        assert v % PO.INSTANCE_OFFSET == hf_label[hf_id]
    fused_hf = {s['label_id'] for s in segments if s['was_fused']}
    assert fused_hf == {v for v in our_ids if num_things <= v < C}


# ---------------------------------------------------------------- mmdet semantics, hand-built

C, NT = 10, 6          # classes 0..5 things, 6..9 stuff, 10 void


@pytest.mark.parametrize('lost,kept', [(21, False), (20, True), (19, True)])
def test_overlap_ratio_around_iou_thr(lost, kept):
    """q0 (thing 2) covers 100 pixels; q1 (thing 4, higher score) takes `lost` of them: ratio (100 - lost) / 100 against
    iou_thr 0.8 -- 0.79 drops q0, 0.80 (not < 0.8) and 0.81 keep it."""
    probs = planted_probs([(2, 0.9), (4, 0.95)], C)
    m = strip((0, 100), (100 - lost, 200))
    pan, st = PO.panoptic_postprocess(probs, m, NT)
    assert st['mask_area'].tolist() == [100 - lost, 100 + lost]
    assert st['original_area'].tolist() == [100, 100 + lost]
    row = pan[0]
    if kept:
        assert (row[:100 - lost] == 2 + 1000).all() and (row[100 - lost:] == 4 + 2000).all()
    else:
        assert (row[:100 - lost] == C).all() and (row[100 - lost:] == 4 + 1000).all()
    # hf_semantics drops at ratio <= thr: the 0.80 case flips there
    pan_hf, _ = PO.panoptic_postprocess(probs, m, NT, hf_semantics=True)
    assert bool((pan_hf[0, :100 - lost] != C).all()) == (lost < 20)


@pytest.mark.parametrize('filter_low_score', [False, True])
def test_filter_low_score_and_mask_area_larger_than_filtered_mask(filter_low_score):
    """One kept query wins every pixel (mask_area 200) but has sigmoid >= 0.5 on only 100 (original_area 100): the
    ratio 2 passes; filter_low_score restricts the painted pixels to the 100."""
    probs = planted_probs([(3, 0.9)], C)
    pan, st = PO.panoptic_postprocess(probs, strip((0, 100)), NT, filter_low_score=filter_low_score)
    assert st['mask_area'].tolist() == [200] and st['original_area'].tolist() == [100]
    assert (pan[0, :100] == 1003).all()
    assert (pan[0, 100:] == (C if filter_low_score else 1003)).all()


def test_no_kept_query_leaves_void():
    # void winner, a score below the threshold, and a score equal to fp32(0.8) (not > 0.800000011920929)
    probs = planted_probs([(C, 0.99), (1, 0.5), (2, 0.8)], C)
    pan, st = PO.panoptic_postprocess(probs, strip((0, 200), (0, 200), (0, 200)), NT)
    assert not st['keep'].any() and (pan == C).all()


def test_two_stuff_queries_merge_and_do_not_consume_instance_ids():
    probs = planted_probs([(7, 0.9), (1, 0.9), (7, 0.9)], C)
    pan, st = PO.panoptic_postprocess(probs, strip((0, 60), (60, 120), (120, 200)), NT)
    assert (pan[0, :60] == 7).all() and (pan[0, 120:] == 7).all()
    assert (pan[0, 60:120] == 1001).all()                            # the only thing: instance id 1
    assert st['seg_value'].tolist() == [7, 1001, 7]


def test_thing_ids_skip_dropped_queries():
    """q1 loses most of its area to q2 and is dropped; q2 and q3 get ids 2 and 3 (q0 has 1)."""
    probs = planted_probs([(0, 0.9), (1, 0.85), (2, 0.95), (5, 0.9)], C)
    pan, st = PO.panoptic_postprocess(probs, strip((0, 50), (50, 100), (60, 150), (150, 200)), NT)
    assert st['seg_value'].tolist() == [1000, -1, 2002, 3005]
    assert (pan[0, :50] == 1000).all() and (pan[0, 50:60] == C).all()
    assert (pan[0, 60:150] == 2002).all() and (pan[0, 150:] == 3005).all()


def test_exact_tie_goes_to_the_lower_kept_index():
    probs = planted_probs([(C, 0.9), (4, 0.9), (5, 0.9)], C)          # q0 not kept: kept indices are q1 -> 0, q2 -> 1
    m = strip((0, 0), (0, 200), (0, 200))
    pan, st = PO.panoptic_postprocess(probs, m, NT)
    assert (pan == 1004).all()
    assert st['mask_area'].tolist() == [0, 200, 0] and st['seg_value'].tolist() == [-1, 1004, -1]


def test_resample_chain_shapes():
    lowres = torch.randn((3, 16, 20))
    meta = dict(batch_input_shape=(64, 80), img_shape=(60, 77, 3), ori_shape=(90, 115, 3))
    assert PO.resample_logits(lowres, meta['batch_input_shape'], meta['img_shape']).shape == (3, 60, 77)
    assert PO.resample_logits(lowres, meta['batch_input_shape'], meta['img_shape'], meta['ori_shape']).shape == (3, 90, 115)
