"""The matching-based losses of the training step (SURVEY.md section 8 row f2): `loss_single` of the reference
(open_set/models/mask2former_head.py:464-629) without its grounding / caption terms -- target assignment by Hungarian
matching on point-sampled masks (`_get_target_single`, :320-390; open_set/assigners/mask_hungarian_assigner.py:47-146),
the class-weighted cross entropies loss_cls / loss_cls_emb (:520-538) and the importance-sampled point losses loss_mask /
loss_dice (:600-627).

The reference reaches into mmcv / mmdet for every step (mmcv.ops.point_sample, mmdet's match costs, DiceLoss,
CrossEntropyLoss, get_uncertain_point_coords_with_randomness); here the sampling, the cost matrix and the losses with their
backward are kernels of the C-ABI library (csrc/match_kernels.cu).  What stays with the host / torch, exactly as in the
reference: the Hungarian solve (scipy's linear_sum_assignment on the (Q, G) cost matrix, assigner :127-134), the random
point draws (torch.rand) and the top-k of the uncertainty sampling.

Panoptic targets (mmdet MaskFormerHead.preprocess_gt, :903) are kept compact: `preprocess_gt` uploads the unpadded things
masks and finds each semantic map's stuff labels on the device, and the targets are only ever point-sampled from there
(`PanopticTargets`); no (G, Hp, Wp) mask tensor exists.

`MatchingLosses` plugs into `Mask2FormerHeadOpenB200.matching_losses` (head.py `loss`), which merges its dict with the
grounding terms: together they are the reference's full loss dict (caption generation excepted, row f4)."""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import lib as _lib

EPS32 = float(torch.finfo(torch.float32).eps)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _ctx(t):
    from .grounding import _Handle
    lib, h = _Handle.get(t.device)
    return lib, h, C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


class _PointSample(torch.autograd.Function):
    """mmcv.ops.point_sample for one-channel maps: inp (N, H, W), coords (N or 1, P, 2) -> (N, P)."""

    @staticmethod
    def forward(ctx, inp, coords):
        if not inp.is_cuda:
            raise _lib.CggError('point_sample runs on a CUDA device only (no CPU path)')
        inp = inp.float().contiguous()
        coords = coords.float().contiguous()
        N, H, W = inp.shape
        P = coords.shape[1]
        shared = int(coords.shape[0] == 1 and N != 1)
        assert coords.shape[0] in (1, N)
        out = torch.empty((N, P), dtype=torch.float32, device=inp.device)
        lib, h, s = _ctx(inp)
        _lib.check(lib.cgg_point_sample(h, _p(inp), _p(coords), _p(out), N, H, W, P, shared, s), h, 'cgg_point_sample')
        ctx.save_for_backward(coords)
        ctx.shape, ctx.shared = (N, H, W), shared
        return out

    @staticmethod
    def backward(ctx, g):
        (coords,) = ctx.saved_tensors
        N, H, W = ctx.shape
        g = g.contiguous()
        din = torch.empty((N, H, W), dtype=torch.float32, device=g.device)
        lib, h, s = _ctx(g)
        _lib.check(lib.cgg_point_sample_backward(h, _p(g), _p(coords), _p(din), N, H, W, coords.shape[1], ctx.shared, s), h,
                   'cgg_point_sample_backward')
        return din, None


def point_sample(inp, coords):
    return _PointSample.apply(inp, coords)


class _PointLosses(torch.autograd.Function):
    """(dice_rows, bce_rows) of matched rows: 1 - dice(sigmoid(pred), t) and sum_p BCE-with-logits(pred, t)."""

    @staticmethod
    def forward(ctx, pred, target, eps):
        pred, target = pred.contiguous(), target.contiguous()
        N, P = pred.shape
        abc = torch.empty((N, 3), dtype=torch.float32, device=pred.device)
        dice = torch.empty((N,), dtype=torch.float32, device=pred.device)
        bce = torch.empty((N,), dtype=torch.float32, device=pred.device)
        lib, h, s = _ctx(pred)
        _lib.check(lib.cgg_point_losses(h, _p(pred), _p(target), N, P, float(eps), _p(abc), _p(dice), _p(bce), s), h,
                   'cgg_point_losses')
        ctx.save_for_backward(pred, target, abc)
        ctx.eps = float(eps)
        return dice, bce

    @staticmethod
    def backward(ctx, g_dice, g_bce):
        pred, target, abc = ctx.saved_tensors
        N, P = pred.shape
        dx = torch.empty_like(pred)
        lib, h, s = _ctx(pred)
        gd, gb = g_dice.contiguous(), g_bce.contiguous()      # named: a temporary freed inside the call would be recycled
        _lib.check(lib.cgg_point_losses_backward(h, _p(pred), _p(target), _p(abc), N, P, ctx.eps, _p(gd), _p(gb), _p(dx), s),
                   h, 'cgg_point_losses_backward')
        return dx, None, None


class _WeightedCE(torch.autograd.Function):
    """row_loss = w[label] * CE(logits, label) per row (F.cross_entropy(weight=w, reduction='none')), plus w[label]."""

    @staticmethod
    def forward(ctx, logits, labels, class_weight):
        logits = logits.float().contiguous()
        R, C1 = logits.shape
        row_loss = torch.empty((R,), dtype=torch.float32, device=logits.device)
        row_w, lse = torch.empty_like(row_loss), torch.empty_like(row_loss)
        lib, h, s = _ctx(logits)
        _lib.check(lib.cgg_weighted_ce(h, _p(logits), _p(labels), _p(class_weight), R, C1, _p(row_loss), _p(row_w), _p(lse), s),
                   h, 'cgg_weighted_ce')
        ctx.save_for_backward(logits, labels, class_weight, lse)
        ctx.mark_non_differentiable(row_w)
        return row_loss, row_w

    @staticmethod
    def backward(ctx, g, _gw):
        logits, labels, class_weight, lse = ctx.saved_tensors
        R, C1 = logits.shape
        d = torch.empty_like(logits)
        lib, h, s = _ctx(logits)
        g = g.contiguous()
        _lib.check(lib.cgg_weighted_ce_backward(h, _p(logits), _p(labels), _p(class_weight), _p(lse), R, C1, _p(g), _p(d), s),
                   h, 'cgg_weighted_ce_backward')
        return d, None, None


def matching_cost(mask_points, gt_points, gt_labels, cls_scores=None, cls_emb_logits=None, w_cls=0.0, w_cls_emb=2.0,
                  w_mask=5.0, w_dice=5.0, dice_eps=1.0):
    """(Q, G) Hungarian cost of mask_hungarian_assigner.py:98-125 from the point-sampled logits (Q, P) / masks (G, P)."""
    Q, P = mask_points.shape
    G = gt_points.shape[0]
    cost = torch.empty((Q, G), dtype=torch.float32, device=mask_points.device)
    if Q == 0 or G == 0:
        return cost
    ref = cls_emb_logits if cls_emb_logits is not None else cls_scores
    C1 = ref.shape[-1] if ref is not None else 1
    scratch = torch.empty((4 * Q + G,), dtype=torch.float32, device=mask_points.device)
    lib, h, s = _ctx(mask_points)
    # every converted operand keeps a name until the call has been issued (a temporary would be recycled by the allocator)
    x, g = mask_points.float().contiguous(), gt_points.float().contiguous()
    cls = cls_scores.float().contiguous() if (cls_scores is not None and w_cls != 0) else None
    emb = cls_emb_logits.float().contiguous() if (cls_emb_logits is not None and w_cls_emb != 0) else None
    lab = gt_labels.long().contiguous()
    _lib.check(lib.cgg_matching_cost(h, _p(x), _p(g), _p(cls), _p(emb), _p(lab), Q, G, C1, P,
                                     float(w_cls if cls is not None else 0.0), float(w_cls_emb if emb is not None else 0.0),
                                     float(w_mask), float(w_dice), float(dice_eps), _p(scratch), _p(cost), s), h,
               'cgg_matching_cost')
    return cost


class PanopticTargets:
    """Compact panoptic training targets of a batch, from `preprocess_gt`: per image the unpadded things planes (uint8),
    the semantic map and its stuff labels, described by one cgg_gt_image per image in device memory.  Target g of image i
    is things plane g (zero outside the plane, up to the image's pad_shape) for g < num_things[i], else the stuff mask
    `sem_i == stuff label`; targets are only ever point-sampled, bit for bit as `point_sample` samples the dense padded
    masks of mmdet's preprocess_gt."""

    def __init__(self, images, rows, num_gts, keep):
        self.images = images            # B cgg_gt_image descriptors (device bytes)
        self.rows = rows                # (sum G, 2) int32 (image, target), every target of the batch in image order
        self.num_gts = num_gts          # per image, things + stuff (host ints)
        self._keep = keep               # the buffers the descriptors point into

    def __len__(self):
        return len(self.num_gts)

    def _sample(self, rows, coords, per_image):
        c = coords.float().contiguous()
        R, P = rows.shape[0], c.shape[1]
        out = torch.empty((R, P), dtype=torch.float32, device=c.device)
        if R == 0 or P == 0:
            return out
        lib, h, s = _ctx(c)
        _lib.check(lib.cgg_gt_point_sample(h, _p(self.images), _p(rows), _p(c), _p(out), R, P, int(per_image), s), h,
                   'cgg_gt_point_sample')
        return out

    def sample_shared(self, coords):
        """Every target of image i at the points coords[i] (B, P, 2) -> (sum G, P), images in order (the cost matrices)."""
        return self._sample(self.rows, coords, True)

    def sample_rows(self, rows, coords):
        """Row r of `rows` (N, 2) int32 = (image, target) at its own points coords[r] (N, P, 2) -> (N, P) (loss targets)."""
        return self._sample(rows.int().contiguous(), coords, False)


def _is_bitmap_masks(m):
    return hasattr(m, 'masks') and hasattr(m, 'height') and hasattr(m, 'width')


def check_stuff_extent(num_stuff, img_metas, sem_hw):
    """mmdet concatenates the things masks (padded to pad_shape) with the stuff masks (the semantic map's shape): that
    fails when the two extents differ and the image has a stuff target."""
    for i, n in enumerate(num_stuff):
        pad = tuple(int(v) for v in img_metas[i]['pad_shape'][:2])
        if n > 0 and pad != tuple(sem_hw):
            raise _lib.CggError('image %d: pad_shape %s differs from the semantic map %s, and it has %d stuff targets'
                                % (i, pad, tuple(sem_hw), n))


def stuff_labels(sem, num_things, num_stuff):
    """The stuff labels present in each semantic map of sem (B, 1, Hs, Ws) (uint8 or int64, on the device), in
    [num_things, num_things + num_stuff) -> (labels (B, num_stuff) int64 ascending, -1 past the count; counts (B,) int32)."""
    sem = sem.contiguous()
    B, Hs, Ws = sem.shape[0], sem.shape[-2], sem.shape[-1]
    labels = torch.empty((B, num_stuff), dtype=torch.long, device=sem.device)
    counts = torch.zeros((B,), dtype=torch.int32, device=sem.device)
    if num_stuff == 0:
        return labels, counts
    bitmap = torch.empty((B * ((num_stuff + 31) // 32),), dtype=torch.int32, device=sem.device)
    lib, h, s = _ctx(sem)
    _lib.check(lib.cgg_panoptic_stuff_labels(h, _p(sem), int(sem.dtype == torch.int64), B, Hs, Ws, num_things,
                                             num_things + num_stuff, _p(bitmap), _p(labels), _p(counts), s), h,
               'cgg_panoptic_stuff_labels')
    return labels, counts


def preprocess_gt(gt_labels_list, gt_masks_list, gt_semantic_segs, img_metas, num_things, num_stuff, device):
    """mmdet 2.28.2 MaskFormerHead.preprocess_gt / preprocess_panoptic_gt, compact: -> (labels_list, PanopticTargets).
    labels: int64 on `device`, things then the stuff labels present in the semantic map, ascending.  gt_masks_list[i]:
    mmdet BitmapMasks (anything with `.masks` (G, h, w), `.height`, `.width`; uploaded unpadded through one pinned
    staging buffer) or a bool / uint8 (G, h, w) tensor; padded implicitly to img_metas[i]['pad_shape'].  gt_semantic_segs:
    None (things only) or the (B, 1, Hs, Ws) batch (a list of (1, Hs, Ws) maps is stacked), uint8 or int64, pad value 255."""
    B = len(gt_labels_list)
    if len(gt_masks_list) != B or len(img_metas) != B:
        raise _lib.CggError('preprocess_gt: %d label lists, %d mask lists, %d img_metas' % (B, len(gt_masks_list), len(img_metas)))
    device = torch.device(device)
    planes = []                                                    # per image: (numpy array or device tensor, G, h, w)
    for i, (lab, m) in enumerate(zip(gt_labels_list, gt_masks_list)):
        if _is_bitmap_masks(m):
            arr = np.asarray(m.masks)
            h, w = int(m.height), int(m.width)
            arr = arr.reshape(-1, h, w) if arr.size else np.zeros((0, h, w), np.uint8)
            arr = np.ascontiguousarray(arr if arr.dtype in (np.uint8, np.bool_) else arr != 0).view(np.uint8)
        elif torch.is_tensor(m):
            if m.dtype not in (torch.bool, torch.uint8) or m.dim() != 3:
                raise _lib.CggError('image %d: a mask tensor must be bool or uint8 (G, h, w), got %s %s' % (i, m.dtype, tuple(m.shape)))
            arr = m
        else:
            raise _lib.CggError('image %d: masks must be mmdet BitmapMasks or a (G, h, w) tensor, got %s' % (i, type(m).__name__))
        G, h, w = (int(v) for v in arr.shape)
        if G != int(lab.shape[0]):
            raise _lib.CggError('image %d: %d masks for %d labels' % (i, G, int(lab.shape[0])))
        pad_h, pad_w = (int(v) for v in img_metas[i]['pad_shape'][:2])
        if h > pad_h or w > pad_w:
            raise _lib.CggError('image %d: masks (%d, %d) larger than pad_shape (%d, %d)' % (i, h, w, pad_h, pad_w))
        planes.append((arr, G, h, w, pad_h, pad_w))
    sem = None
    if gt_semantic_segs is not None:
        sem = gt_semantic_segs if torch.is_tensor(gt_semantic_segs) else torch.stack([torch.as_tensor(x) for x in gt_semantic_segs])
        if sem.dtype not in (torch.uint8, torch.int64):
            raise _lib.CggError('gt_semantic_seg must be uint8 or int64, got %s' % sem.dtype)
        if sem.dim() != 4 or sem.shape[0] != B or sem.shape[1] != 1:
            raise _lib.CggError('gt_semantic_seg must be (B, 1, Hs, Ws), got %s' % (tuple(sem.shape),))
    labels = [torch.as_tensor(x).to(device=device, dtype=torch.long) for x in gt_labels_list]
    keep = []
    n_stuff = [0] * B
    if sem is not None:
        sem = sem.to(device).contiguous()
        Hs, Ws = int(sem.shape[2]), int(sem.shape[3])
        stuff, counts = stuff_labels(sem, num_things, num_stuff)
        n_stuff = counts.tolist()                                  # the batch's one read-back: it shapes the cost matrices
        check_stuff_extent(n_stuff, img_metas, (Hs, Ws))
        labels = [torch.cat((labels[i], stuff[i, :n_stuff[i]])) for i in range(B)]
        keep += [sem, stuff]
    # one staging buffer, one copy: B descriptors, the (image, target) table, then every host-side things plane
    desc_bytes = B * C.sizeof(_lib.GtImage)
    num_gts = [p[1] + n for p, n in zip(planes, n_stuff)]
    rows = np.array([(i, g) for i in range(B) for g in range(num_gts[i])], dtype=np.int32).reshape(-1, 2)
    at = desc_bytes + rows.nbytes
    offsets = []
    for arr, G, h, w, _, _ in planes:
        offsets.append(at if isinstance(arr, np.ndarray) else None)
        at += arr.nbytes if isinstance(arr, np.ndarray) else 0
    buf = torch.empty((at,), dtype=torch.uint8, device=device)
    staging = torch.empty((at,), dtype=torch.uint8, pin_memory=True)
    st = staging.numpy()
    descs = (_lib.GtImage * B)()
    elem = sem.element_size() if sem is not None else 0
    for i, ((arr, G, h, w, pad_h, pad_w), off) in enumerate(zip(planes, offsets)):
        d = descs[i]
        if off is not None:
            st[off:off + arr.nbytes] = arr.reshape(-1)
            d.things = buf.data_ptr() + off
        else:
            t = arr.to(device).contiguous().view(torch.uint8)
            keep.append(t)
            d.things = t.data_ptr()
        d.num_things, d.h, d.w, d.pad_h, d.pad_w = G, h, w, pad_h, pad_w
        if n_stuff[i]:
            d.sem = sem.data_ptr() + i * Hs * Ws * elem
            d.sem_stride, d.sem_is_i64 = Ws, int(sem.dtype == torch.int64)
            d.stuff_labels = stuff.data_ptr() + i * num_stuff * 8
            d.num_stuff = n_stuff[i]
    st[:desc_bytes] = np.frombuffer(bytes(descs), dtype=np.uint8)
    st[desc_bytes:desc_bytes + rows.nbytes] = rows.reshape(-1).view(np.uint8)
    buf.copy_(staging, non_blocking=True)                          # a plain cudaMemcpyAsync from pinned memory
    keep += [buf, staging]
    images = buf[:desc_bytes]
    rows_dev = buf[desc_bytes:desc_bytes + rows.nbytes].view(torch.int32).view(-1, 2)
    return labels, PanopticTargets(images, rows_dev, num_gts, keep)


def _reduce_mean(t):
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        t = t.clone()
        dist.all_reduce(t.div_(dist.get_world_size()))
    return t


class MatchingLosses:
    """Callable for `head.matching_losses`: (all_cls_scores, all_cls_emb_preds, all_mask_preds, gt_labels_list,
    gt_masks_list, img_metas) -> dict with loss_cls / loss_cls_emb / loss_mask / loss_dice of the last head call and
    `d{i}.`-prefixed copies for the others (head.py:437-461).  Configuration follows the reference's config keys
    (configs/openset_panoptic/coco_panoptic_p20.py:111-139, :163-175)."""

    def __init__(self, head, train_cfg=None, loss_cls=None, loss_cls_emb=None, loss_mask=None, loss_dice=None):
        tc = dict(train_cfg or {})
        self.head = head
        self.num_points = int(tc.get('num_points', 12544))
        self.oversample_ratio = float(tc.get('oversample_ratio', 3.0))
        self.importance_sample_ratio = float(tc.get('importance_sample_ratio', 0.75))
        a = dict(tc.get('assigner', {}) or {})
        g = lambda d, k, default: (dict(d.get(k) or {})).get('weight', default)       # noqa: E731
        self.w_cls, self.w_cls_emb = g(a, 'cls_cost', 0.0), g(a, 'cls_emb_cost', 2.0)
        self.w_mask, self.w_dice = g(a, 'mask_cost', 5.0), g(a, 'dice_cost', 5.0)
        self.cost_dice_eps = (dict(a.get('dice_cost') or {})).get('eps', 1.0)
        lc, le = dict(loss_cls or {}), dict(loss_cls_emb or {})
        lm, ld = dict(loss_mask or {}), dict(loss_dice or {})
        self.loss_cls_weight = lc.get('loss_weight', 0.0)
        self.loss_cls_emb_weight = le.get('loss_weight', 2.0)
        self.loss_mask_weight = lm.get('loss_weight', 5.0)
        self.loss_dice_weight = ld.get('loss_weight', 5.0)
        self.dice_eps = ld.get('eps', 1.0)
        ncls = head.num_classes
        self.class_weight = torch.tensor(lc.get('class_weight') or ([1.0] * ncls + [0.1]), dtype=torch.float32)
        self.rand = lambda *shape, device=None: torch.rand(*shape, device=device)      # tests swap in a seeded CPU stream

    # ---- targets (mask2former_head.py:320-390)
    @torch.no_grad()
    def get_target_single(self, cls_score, cls_emb_logit, mask_pred, gt_labels, gt_masks):
        """gt_masks: the dense (G, H, W) masks, whose matched rows are returned, or a one-image PanopticTargets, whose
        matched target indices are returned."""
        dev = mask_pred.device
        G = gt_labels.shape[0]
        coords = self.rand(1, self.num_points, 2, device=dev).to(dev)
        if isinstance(gt_masks, PanopticTargets):
            if len(gt_masks) != 1:
                raise _lib.CggError('get_target_single takes the targets of one image, got %d' % len(gt_masks))
            labels, pos_gt, mask_weights, n = self._assign(cls_score, cls_emb_logit, mask_pred, gt_labels,
                                                           gt_masks.sample_shared(coords), coords)
            return labels, pos_gt, mask_weights, n
        if G == 0:
            labels, _, mask_weights, _ = self._assign(cls_score, cls_emb_logit, mask_pred, gt_labels, None, coords)
            return labels, gt_masks[:0], mask_weights, 0
        labels, pos_gt, mask_weights, n = self._assign(cls_score, cls_emb_logit, mask_pred, gt_labels,
                                                       point_sample(gt_masks.float(), coords), coords)
        return labels, gt_masks[pos_gt], mask_weights, n

    @torch.no_grad()
    def _assign(self, cls_score, cls_emb_logit, mask_pred, gt_labels, gt_points, coords):
        """One image's Hungarian assignment from its targets sampled at coords (None or no row: no target) ->
        (labels (Q,), matched target indices in query order, mask_weights (Q,), number matched)."""
        dev = mask_pred.device
        Q = mask_pred.shape[0]
        labels = torch.full((Q,), self.head.num_classes, dtype=torch.long, device=dev)
        mask_weights = torch.zeros((Q,), dtype=torch.float32, device=dev)
        if gt_points is None or gt_points.shape[0] == 0:
            return labels, torch.zeros((0,), dtype=torch.long, device=dev), mask_weights, 0
        mask_points = point_sample(mask_pred.detach(), coords)
        cost = matching_cost(mask_points, gt_points, gt_labels, cls_score.detach(),
                             None if cls_emb_logit is None else cls_emb_logit.detach(), self.w_cls, self.w_cls_emb, self.w_mask,
                             self.w_dice, self.cost_dice_eps)
        from scipy.optimize import linear_sum_assignment
        rows, cols = linear_sum_assignment(cost.cpu().numpy())           # on the host, as in the reference (:127-134)
        order = rows.argsort()                                           # MaskPseudoSampler: positives in query order
        pos = torch.from_numpy(rows[order]).to(dev)
        pos_gt = torch.from_numpy(cols[order]).to(dev)
        labels[pos] = gt_labels[pos_gt]
        mask_weights[pos] = 1.0
        return labels, pos_gt, mask_weights, int(pos.numel())

    @torch.no_grad()
    def _targets_compact(self, cls_scores, cls_emb_logits, mask_preds, gt_labels_list, targets):
        """get_target_single for every image of PanopticTargets, with all the cost matrices' ground truth sampled in one
        launch -> (labels (B*Q,), mask_weights (B, Q), number matched, matched (image, target) rows in query order)."""
        B = cls_scores.shape[0]
        dev = cls_scores.device
        if len(targets) != B:
            raise _lib.CggError('%d images of targets for a batch of %d' % (len(targets), B))
        # get_target_single's point draws, in the same order: no other draw falls between them
        coords = [self.rand(1, self.num_points, 2, device=dev).to(dev) for _ in range(B)]
        gt_points = targets.sample_shared(torch.cat(coords, 0))
        labels, weights, rows, num_pos, at = [], [], [], 0, 0
        for i in range(B):
            G = targets.num_gts[i]
            lab, pos_gt, mw, n = self._assign(cls_scores[i], None if cls_emb_logits is None else cls_emb_logits[i],
                                              mask_preds[i], gt_labels_list[i].to(dev), gt_points[at:at + G], coords[i])
            at += G
            labels.append(lab), weights.append(mw), rows.append(torch.stack((torch.full_like(pos_gt, i), pos_gt), 1))
            num_pos += n
        return torch.stack(labels, 0).flatten(), torch.stack(weights, 0), num_pos, torch.cat(rows, 0).int()

    def uncertain_point_coords(self, mask_preds):
        """mmdet get_uncertain_point_coords_with_randomness on (N, h, w) logits -> (N, num_points, 2)."""
        N = mask_preds.shape[0]
        dev = mask_preds.device
        num_sampled = int(self.num_points * self.oversample_ratio)
        coords = self.rand(N, num_sampled, 2, device=dev).to(dev)
        unc = -point_sample(mask_preds, coords).abs()
        num_uncertain = int(self.importance_sample_ratio * self.num_points)
        num_random = self.num_points - num_uncertain
        idx = torch.topk(unc, k=num_uncertain, dim=1)[1]
        picked = torch.gather(coords, 1, idx.unsqueeze(-1).expand(-1, -1, 2))
        if num_random > 0:
            picked = torch.cat((picked, self.rand(N, num_random, 2, device=dev).to(dev)), dim=1)
        return picked

    # ---- one head call (mask2former_head.py:464-629 without the caption terms)
    def loss_single(self, cls_scores, cls_emb_logits, mask_preds, gt_labels_list, gt_masks_list):
        """gt_masks_list: per image dense (G, H, W) masks, or the batch's PanopticTargets (preprocess_gt)."""
        B, Q = cls_scores.shape[:2]
        dev = cls_scores.device
        compact = isinstance(gt_masks_list, PanopticTargets)
        if compact:
            labels, mask_weights, num_pos, target_rows = self._targets_compact(cls_scores, cls_emb_logits, mask_preds,
                                                                               gt_labels_list, gt_masks_list)
        else:
            labels, targets, weights, num_pos = [], [], [], 0
            for i in range(B):
                lab, mt, mw, n = self.get_target_single(cls_scores[i], None if cls_emb_logits is None else cls_emb_logits[i],
                                                        mask_preds[i], gt_labels_list[i].to(dev), gt_masks_list[i].to(dev))
                labels.append(lab), targets.append(mt), weights.append(mw)
                num_pos += n
            labels = torch.stack(labels, 0).flatten()
            mask_targets = torch.cat(targets, 0)
            mask_weights = torch.stack(weights, 0)
        cw = self.class_weight.to(dev)
        out = {}
        row_loss, row_w = _WeightedCE.apply(cls_scores.flatten(0, 1), labels, cw)
        avg = row_w.sum() + EPS32
        out['loss_cls'] = self.loss_cls_weight * row_loss.sum() / avg
        out['loss_cls_emb'] = cls_scores.new_tensor(0.0)
        if cls_emb_logits is not None:
            row_loss_e, _ = _WeightedCE.apply(cls_emb_logits.flatten(0, 1), labels, cw)
            out['loss_cls_emb'] = self.loss_cls_emb_weight * row_loss_e.sum() / avg
        num_total = float(max(float(_reduce_mean(torch.tensor([float(num_pos)], device=dev))), 1.0))
        pos_preds = mask_preds[mask_weights > 0]
        if (target_rows if compact else mask_targets).shape[0] == 0:     # zero match (:582-586)
            out['loss_dice'] = pos_preds.sum()
            out['loss_mask'] = pos_preds.sum()
            return out, labels.view(B, Q), mask_weights
        with torch.no_grad():
            coords = self.uncertain_point_coords(pos_preds.detach())
            if compact:
                point_targets = gt_masks_list.sample_rows(target_rows, coords)
            else:
                point_targets = point_sample(mask_targets.float(), coords)
        point_preds = point_sample(pos_preds, coords)
        dice_rows, bce_rows = _PointLosses.apply(point_preds, point_targets, self.dice_eps)
        out['loss_dice'] = self.loss_dice_weight * dice_rows.sum() / (num_total + EPS32)
        out['loss_mask'] = self.loss_mask_weight * bce_rows.sum() / (num_total * self.num_points + EPS32)
        return out, labels.view(B, Q), mask_weights

    def __call__(self, all_cls_scores, all_cls_emb_preds, all_mask_preds, gt_labels_list, gt_masks_list, img_metas=None):
        from .grounding import similarity
        head = self.head
        n = len(all_cls_scores)
        losses = {}
        for j in range(n):
            if getattr(head, 'loss_only_last', False) and j != n - 1:
                continue
            logits = None
            if head.use_class_emb:                                       # _get_cls_emb_logits, head.py:631-648
                B, Q, D = all_cls_emb_preds[j].shape
                logits = similarity(all_cls_emb_preds[j].reshape(B * Q, D), head.class_embs,
                                    1.0 / float(head.softmax_temperature)).view(B, Q, -1)
            out, _, _ = self.loss_single(all_cls_scores[j], logits, all_mask_preds[j], gt_labels_list, gt_masks_list)
            prefix, scale = ('', 1.0) if j == n - 1 else ('d%d.' % j, getattr(head, 'loss_aux_weight', 1.0))
            for k, v in out.items():
                losses[prefix + k] = v * scale
        return losses
