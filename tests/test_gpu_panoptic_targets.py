"""GPU tests of the compact panoptic training targets (cgg_b200/matching.py `preprocess_gt`, `PanopticTargets`;
csrc/match_kernels.cu stuff_presence / stuff_compact / gt_point_sample kernels) against the dense targets of the oracle's
restatement of mmdet 2.28.2 preprocess_gt (oracle/panoptic_targets_oracle.py).  The random point draws come from the
same seeded CPU torch.rand stream on both sides, so the compact path must reproduce the dense one bit for bit."""
import numpy as np
import pytest
import torch

from oracle import matching_oracle as MO
from oracle import panoptic_targets_oracle as PT
from cgg_b200 import synth, matching
from cgg_b200.head import build_head_from_state_dict
from cgg_b200.lib import CggError

pytestmark = pytest.mark.gpu
DEV = 'cuda'
NT, NS = 30, 18                    # 48 classes, the last 18 stuff


class Bitmap:
    """The part of mmdet's BitmapMasks that preprocess_gt reads."""

    def __init__(self, masks):
        self.masks = np.asarray(masks, dtype=np.uint8)
        self.height, self.width = self.masks.shape[1:]


def make_targets(seed, things=(3, 0, 2), stuff=(2, 1, 0), pad=(40, 52), sem_dtype=torch.uint8, bitmap=True):
    """Per image: `things` random masks of an image smaller than `pad`, and a semantic map (pad) with `stuff` stuff
    segments, thing-label pixels, out-of-range labels and the 255 padding."""
    g = torch.Generator().manual_seed(seed)
    B = len(things)
    labels, masks, metas = [], [], []
    sem = torch.full((B, 1) + pad, 255, dtype=sem_dtype)
    for b in range(B):
        h, w = pad[0] - 3 - b, pad[1] - 5 - 2 * b
        m = (torch.rand((things[b], h, w), generator=g) > 0.6).to(torch.uint8)
        labels.append(torch.randint(0, NT, (things[b],), generator=g))
        masks.append(Bitmap(m.numpy()) if bitmap else m.bool().to(DEV))
        metas.append(dict(pad_shape=pad + (3,)))
        sem[b, 0, :h, :w] = torch.randint(0, NT, (h, w), generator=g).to(sem_dtype)      # thing pixels: no target
        sem[b, 0, 0, :3] = NT + NS                                                    # == num_classes: no target
        for k, lab in enumerate(torch.randperm(NS, generator=g)[:stuff[b]].tolist()):
            y0, x0 = int(torch.randint(0, pad[0] - 8, (1,), generator=g)), int(torch.randint(0, pad[1] - 8, (1,), generator=g))
            sem[b, 0, y0:y0 + 4 + 3 * k, x0:x0 + 5 + k] = NT + lab
    return labels, masks, sem, metas


def dense(labels, masks, sem, metas):
    mm = [torch.from_numpy(m.masks) if isinstance(m, Bitmap) else m.cpu() for m in masks]
    return PT.preprocess_gt(labels, mm, None if sem is None else sem.cpu(), metas, NT, NS)


@pytest.fixture(scope='module')
def head():
    return build_head_from_state_dict(synth.make_params(seed=2, num_queries=20), 20, 49, 'fp32', DEV, num_stuff_classes=NS)


def _ml(head, P):
    ml = matching.MatchingLosses(head, train_cfg=dict(num_points=P))
    ml.rand = lambda *shape, device=None: torch.rand(*shape)          # the oracle's stream: seeded CPU generator
    return ml


@pytest.mark.parametrize('dtype', [torch.uint8, torch.int64])
def test_stuff_labels_match_the_oracle_and_cuda_unique_order(dtype):
    g = torch.Generator().manual_seed(5)
    maps = [torch.full((1, 33, 47), 255, dtype=dtype),                         # all padding
            torch.arange(33 * 47).remainder(NT + NS).view(1, 33, 47).to(dtype),  # every stuff class
            torch.randint(0, NT, (1, 33, 47), generator=g).to(dtype),          # things only
            torch.randint(0, 256 if dtype == torch.uint8 else 1000, (1, 33, 47), generator=g).to(dtype)]
    one = torch.full((1, 33, 47), 255, dtype=dtype)
    one[0, 32, 46] = NT + 7                                                   # a 1-pixel segment in the last corner
    maps.append(one)
    sem = torch.stack(maps, 0)
    got, counts = matching.stuff_labels(sem.to(DEV), NT, NS)
    for b in range(sem.shape[0]):
        want = PT.preprocess_panoptic_gt(torch.zeros((0,), dtype=torch.long), torch.zeros((0, 33, 47)), sem[b], NT, NS,
                                         dict(pad_shape=(33, 47)))[0]
        n = int(counts[b])
        assert got[b, :n].cpu().tolist() == want.tolist(), b
        assert (got[b, n:] == -1).all()
        # the reference's order: torch.unique(sorted=False) on a CUDA tensor
        u = torch.unique(sem[b].to(DEV), sorted=False)
        assert got[b, :n].cpu().tolist() == [int(v) for v in u.cpu() if NT <= int(v) < NT + NS], b
    assert counts.tolist()[:2] == [0, NS] and int(counts[4]) == 1


def _coords(g, n, P, pad):
    c = torch.rand((n, P, 2), generator=g) * 1.2 - 0.1                       # some points outside [0, 1]
    c[:, :4] = torch.tensor([[0.0, 0.0], [1.0, 1.0], [0.0, 1.0], [1.0, 0.0]])  # the borders
    k = torch.randint(0, min(pad), (n, 8, 2), generator=g).float()
    c[:, 4:12, 0], c[:, 4:12, 1] = (k[..., 0] + 0.5) / pad[1], (k[..., 1] + 0.5) / pad[0]   # pixel centres
    return c


@pytest.mark.parametrize('sem_dtype,bitmap', [(torch.uint8, True), (torch.int64, False)])
def test_gt_point_sample_is_bit_identical_to_point_sample_of_the_dense_targets(sem_dtype, bitmap):
    labels, masks, sem, metas = make_targets(3, things=(3, 0, 2, 0), stuff=(2, 1, 0, 0), sem_dtype=sem_dtype, bitmap=bitmap)
    d_labels, d_masks = dense(labels, masks, sem, metas)
    got_labels, t = matching.preprocess_gt(labels, masks, sem.to(DEV), metas, NT, NS, DEV)
    assert [x.cpu().tolist() for x in got_labels] == [x.tolist() for x in d_labels]
    assert t.num_gts == [len(x) for x in d_labels] and t.num_gts[0] > 3 and t.num_gts[3] == 0
    g = torch.Generator().manual_seed(4)
    P = 1000
    coords = _coords(g, 4, P, (40, 52)).to(DEV)
    got = t.sample_shared(coords)
    want = torch.cat([matching.point_sample(m.float().to(DEV), coords[i:i + 1]) for i, m in enumerate(d_masks) if m.shape[0]])
    assert torch.equal(got, want)
    rows = torch.tensor([[0, 4], [2, 1], [0, 0], [1, 0], [0, 3], [2, 0]], dtype=torch.int32)
    rc = _coords(g, rows.shape[0], P, (40, 52)).to(DEV)
    got = t.sample_rows(rows.to(DEV), rc)
    want = matching.point_sample(torch.stack([d_masks[i][k] for i, k in rows.tolist()]).float().to(DEV), rc)
    assert torch.equal(got, want)


def _grads_and_losses(ml, a, gt_labels, gt_masks, seed):
    torch.manual_seed(seed)
    got, labels, mw = ml.loss_single(a[0], a[1], a[2], gt_labels, gt_masks)
    sum(got.values()).backward()
    return {k: v.detach().cpu() for k, v in got.items()}, labels.cpu(), mw.cpu(), [x.grad.cpu() for x in a]


@pytest.mark.parametrize('seed,things,stuff', [(1, (3, 2), (2, 1)), (2, (0, 4), (3, 0)), (3, (0, 0), (0, 0)),
                                               (4, (0, 1), (1, 0))])
def test_matching_losses_on_compact_targets_equal_the_dense_ones(head, seed, things, stuff):
    P, Q = 512, 20
    labels, masks, sem, metas = make_targets(seed, things=things, stuff=stuff)
    d_labels, d_masks = dense(labels, masks, sem, metas)
    c_labels, targets = head.preprocess_gt(labels, masks, sem.to(DEV), metas)
    g = torch.Generator().manual_seed(seed)
    B = len(things)
    mask_preds = torch.randn((B, Q, 10, 13), generator=g) * 2
    for b in range(B):                                   # queries correlated with the targets: a real assignment problem
        for k in range(d_masks[b].shape[0]):
            small = torch.nn.functional.interpolate(d_masks[b][k][None, None].float(), size=(10, 13))[0, 0]
            mask_preds[b, (3 * k + b) % Q] += (small * 2 - 1) * 3
    cls = torch.randn((B, Q, NT + NS + 1), generator=g)
    emb = torch.randn((B, Q, NT + NS + 1), generator=g) * 2
    ml = _ml(head, P)
    ml.loss_cls_weight = 0.5
    runs = []
    for lab, gm in ((c_labels, targets), ([x.to(DEV) for x in d_labels], [m.to(DEV) for m in d_masks])):
        a = [t.clone().to(DEV).requires_grad_(True) for t in (cls, emb, mask_preds)]
        runs.append(_grads_and_losses(ml, a, lab, gm, 60 + seed))
    (lc, labc, mwc, gc), (ld, labd, mwd, gd) = runs
    assert torch.equal(labc, labd) and torch.equal(mwc, mwd)
    for k in lc:
        assert torch.equal(lc[k], ld[k]), (k, lc[k], ld[k])
    assert torch.equal(gc[0], gd[0]) and torch.equal(gc[1], gd[1])          # class / embedding logits
    # mask logits: point_sample's backward scatters with atomics, whose order (and so the last bit) varies from run to run
    assert float((gc[2] - gd[2]).abs().max()) <= 1e-6 * float(gd[2].abs().max())
    if sum(things) + sum(stuff) == 0:                    # the zero-match branch
        assert float(lc['loss_mask']) == 0.0 and float(lc['loss_dice']) == 0.0
    # and the oracle's loss_single on the dense targets
    a = [t.clone().requires_grad_(True) for t in (cls, emb, mask_preds)]
    torch.manual_seed(60 + seed)
    want = MO.loss_single_matching(a[0], a[1], a[2], d_labels, d_masks, NT + NS, dict(num_points=P, loss_cls_weight=0.5))
    sum(want[k] for k in ('loss_cls', 'loss_cls_emb', 'loss_mask', 'loss_dice')).backward()
    assert torch.equal(labc, want['labels']) and torch.equal(mwc, want['mask_weights'])
    for k in ('loss_cls', 'loss_cls_emb', 'loss_mask', 'loss_dice'):
        assert abs(float(lc[k]) - float(want[k])) < 2e-5 * max(1.0, abs(float(want[k]))), k
    for x, y in zip(gc, a):
        assert float((x - y.grad).abs().max()) < 1e-4 * float(y.grad.abs().max()) + 1e-9


def test_preprocess_gt_raises_on_a_pad_shape_mismatch_only_with_stuff(head):
    labels, masks, sem, metas = make_targets(8, things=(1, 1), stuff=(0, 2))
    metas[0] = dict(pad_shape=(44, 60, 3))                   # image 0 has no stuff target: accepted
    head.preprocess_gt(labels, masks, sem.to(DEV), metas)
    metas[1] = dict(pad_shape=(44, 60, 3))
    with pytest.raises(CggError, match='stuff targets'):
        head.preprocess_gt(labels, masks, sem.to(DEV), metas)


def _forward_train_losses(head, feats, metas, labels, masks, sem, ids, cmask):
    torch.manual_seed(21)
    head.zero_grad(set_to_none=True)
    losses = head.forward_train(feats, metas, None, labels, masks, sem, list(ids), list(cmask), list(ids), list(cmask))
    sum(losses.values()).backward()
    return {k: v.detach().cpu() for k, v in losses.items()}


def test_forward_train_takes_bitmap_masks_and_the_semantic_map():
    from test_gpu_post import _caption_head
    Q, B = 16, 2
    head, _, _, _ = _caption_head(Q)
    head.num_things_classes, head.num_stuff_classes = NT, NS
    head.train()
    head.matching_losses = _ml(head, 256)
    mf, mems = synth.make_inputs(9, B, 96, 128)
    feats = [mf.to(DEV)] + [m.to(DEV) for m in mems]
    labels, masks, sem, metas = make_targets(11, things=(2, 3), stuff=(3, 1), pad=(96, 128))
    g = torch.Generator().manual_seed(1)
    ids = torch.randint(1000, 1500, (B, 35), generator=g).to(DEV)
    cmask = torch.zeros((B, 35), dtype=torch.long, device=DEV)
    cmask[0, :4] = 1
    cmask[1, :9] = 1
    got = _forward_train_losses(head, feats, metas, labels, masks, sem.to(DEV), ids, cmask)
    want_keys = {p + k for p in [''] + ['d%d.' % i for i in range(9)]
                 for k in ('loss_cls', 'loss_cls_emb', 'loss_mask', 'loss_dice', 'loss_grounding')}
    assert set(got) == want_keys
    d_labels, d_masks = dense(labels, masks, sem, metas)
    want = _forward_train_losses(head, feats, metas, [x.to(DEV) for x in d_labels], [m.to(DEV) for m in d_masks], None,
                                 ids, cmask)
    for k in want_keys:
        assert torch.equal(got[k], want[k]), (k, got[k], want[k])


def test_simple_test_assigns_the_same_labels_from_bitmap_masks():
    from test_gpu_post import _caption_head
    Q = 24
    head, _, _, _ = _caption_head(Q)
    head.eval()
    head.matching_losses = _ml(head, 300)
    mf, mems = synth.make_inputs(12, 1, 128, 160)
    feats = [mf.to(DEV)] + [m.to(DEV) for m in mems]
    g = torch.Generator().manual_seed(3)
    gt_labels = torch.randint(0, 48, (4,), generator=g)
    small = (torch.rand((4, 120, 150), generator=g) > 0.6).to(torch.uint8)      # image size, padded to (128, 160)
    metas = [dict(batch_input_shape=(128, 160), pad_shape=(128, 160, 3))]
    got = []
    for gm in (Bitmap(small.numpy()), PT.pad_masks(small, (128, 160)).long()):
        torch.manual_seed(77)
        with torch.no_grad():
            got.append(head.simple_test(feats, metas, gt_labels=[[gt_labels]], gt_masks=[[gm]])[0].cpu())
    assert torch.equal(got[0], got[1])
