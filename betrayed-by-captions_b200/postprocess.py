"""Test-time step after the decoder path (SURVEY.md section 8f rank 1): the final mask upsample of
`Mask2FormerHeadOpen.simple_test` (open_set/models/mask2former_head.py:957-964) and the instance scoring of
`MaskFormerFusionHeadOpen` (open_set/models/maskformer_fusion_head.py:297-366, :412-425), on the kernels behind
`cgg_upsample_masks`, `cgg_instance_mask_stats`, `cgg_similarity` and `cgg_softmax_rows`.

`instance_postprocess_emb_fused` returns what the reference's `instance_postprocess_emb` returns for every image of the
batch -- labels, boxes with detection scores, binary masks -- but computes the masks' `> 0` bits, pixel counts, sigmoid
sums and bounding boxes in ONE pass over the (B, Q, H/4, W/4) logits: the (B, Q, H, W) fp32 logits that the reference
materialises (6.7 GB for 16 images at 1024^2) never exist.  Masks come back bit-packed (32 pixels per word);
`unpack_masks` expands them when a dense bool tensor is wanted.

`panoptic_postprocess_fused` is the panoptic half (mmdet 2.28.2 `MaskFormerFusionHead.panoptic_postprocess` with the
class-embedding probabilities, behind `cgg_panoptic_fuse`): from the same low-resolution logits it returns the panoptic
map of every image with no host round trip.  `fusion_simple_test` is the fusion head's `simple_test`
(maskformer_fusion_head.py:369-464) on top of both."""
import ctypes as C

import torch

from . import lib as _lib


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _ctx(head, device):
    rt = head._runtime(device)
    return rt, rt.lib, rt.handle, C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def upsample_masks(head, mask_pred, size):
    """F.interpolate(mask_pred, size, mode='bilinear', align_corners=False) -> fp32 (head.py:957-964)."""
    if not mask_pred.is_cuda:
        raise _lib.CggError('upsample_masks runs on CUDA only')
    rt, lib, h, s = _ctx(head, mask_pred.device)
    mp = mask_pred.contiguous()
    B, Q, h4, w4 = mp.shape
    out = torch.empty((B, Q, size[0], size[1]), dtype=torch.float32, device=mp.device)
    assert mp.dtype in (torch.float32, torch.bfloat16)
    _lib.check(lib.cgg_upsample_masks(h, _p(mp), int(mp.dtype == torch.bfloat16), _p(out), B * Q, h4, w4, size[0], size[1], s),
               h, 'cgg_upsample_masks')
    return out


def instance_mask_stats(head, mask_pred, up_size, crops, outs=None, want_bits=True):
    """mask_pred (B, Q, h4, w4) last-call logits; up_size = batch_input_shape; crops[b] = img_shape (h, w); outs[b] =
    ori_shape (h, w) when rescaling (None: no rescale).  Returns dict(bits (B,Q,Hmax,W32) int32 | None, count (B,Q) int32,
    sig_sum (B,Q) fp32, bbox (B,Q,4) int32, out_sizes)."""
    rt, lib, h, s = _ctx(head, mask_pred.device)
    mp = mask_pred.contiguous()
    B, Q, h4, w4 = mp.shape
    outs = outs if outs is not None else crops
    geom = torch.tensor([[c[0], c[1], o[0], o[1]] for c, o in zip(crops, outs)], dtype=torch.int32).to(mp.device)
    Hm, Wm = max(o[0] for o in outs), max(o[1] for o in outs)
    dev = mp.device
    bits = torch.zeros((B, Q, Hm, (Wm + 31) // 32), dtype=torch.int32, device=dev) if want_bits else None
    count = torch.empty((B, Q), dtype=torch.int32, device=dev)
    sig = torch.empty((B, Q), dtype=torch.float32, device=dev)
    bbox = torch.empty((B, Q, 4), dtype=torch.int32, device=dev)
    _lib.check(lib.cgg_instance_mask_stats(h, _p(mp), int(mp.dtype == torch.bfloat16), _p(geom), B, Q, h4, w4, up_size[0],
                                           up_size[1], Hm, Wm, _p(bits), _p(count), _p(sig), _p(bbox), s),
               h, 'cgg_instance_mask_stats')
    return dict(bits=bits, count=count, sig_sum=sig, bbox=bbox, out_sizes=list(outs))


def unpack_masks(bits, width):
    """(..., H, W32) int32 words -> (..., H, width) bool."""
    sh = torch.arange(32, device=bits.device, dtype=torch.int32)
    b = ((bits.unsqueeze(-1) >> sh) & 1).bool()
    return b.flatten(-2)[..., :width]


def cls_emb_scores(head, cls_emb_preds, class_embs):
    """get_cls_emb_scores (maskformer_fusion_head.py:297-315): softmax(emb @ class_embs^T) over the classes."""
    rt, lib, h, s = _ctx(head, cls_emb_preds.device)
    x = cls_emb_preds.reshape(-1, cls_emb_preds.shape[-1])
    scores = rt.similarity(x, class_embs, 1.0)
    _lib.check(lib.cgg_softmax_rows(h, _p(scores), scores.shape[0], scores.shape[1], s), h, 'cgg_softmax_rows')
    return scores.view(*cls_emb_preds.shape[:-1], class_embs.shape[0])


def instance_postprocess_emb_fused(head, mask_cls_emb, mask_pred, class_embs, img_metas, rescale=False, max_per_image=100):
    """`instance_postprocess_emb` (maskformer_fusion_head.py:318-366) for the whole batch, from the LOW-resolution logits.
    mask_cls_emb (B, Q, d_l); mask_pred (B, Q, h4, w4).  Per image: (labels (n,), bboxes (n, 5), packed masks (n, H, W32),
    (H, W))."""
    B, Q = mask_pred.shape[:2]
    up = img_metas[0]['batch_input_shape']
    crops = [m['img_shape'][:2] for m in img_metas]
    outs = [m['ori_shape'][:2] for m in img_metas] if rescale else None
    st = instance_mask_stats(head, mask_pred, up, crops, outs)
    scores_all = cls_emb_scores(head, mask_cls_emb, class_embs)[..., :-1]            # drop the void column
    ncls = scores_all.shape[-1]
    results = []
    for b in range(B):
        sc, top = scores_all[b].flatten().topk(max_per_image, sorted=False)
        labels = top % ncls
        qi = top // ncls
        cnt = st['count'][b, qi].float()
        mask_score = st['sig_sum'][b, qi] / (cnt + 1e-6)
        det = sc * mask_score
        boxes = torch.cat([st['bbox'][b, qi].float(), det[:, None]], dim=-1)
        results.append((labels, boxes, st['bits'][b, qi][:, :st['out_sizes'][b][0]], st['out_sizes'][b]))
    return results


INSTANCE_OFFSET = 1000
_GEOM = {}


def _geom(rows, device):
    """{crop_h, crop_w, out_h, out_w} per image as a device int32 tensor, cached per geometry (a few bytes each, never
    evicted: a captured CUDA graph keeps the pointer).  The first use copies from pinned memory without a host sync; later
    uses, and CUDA-graph captures after a warm-up, copy nothing."""
    key = (device, tuple(rows))
    g = _GEOM.get(key)
    if g is None:
        g = torch.tensor(rows, dtype=torch.int32).pin_memory().to(device, non_blocking=True)
        _GEOM[key] = g
    return g


def panoptic_postprocess_fused(head, probs, mask_pred_lowres, img_metas, rescale=False, test_cfg=None, stats=False):
    """`panoptic_postprocess` (mmdet 2.28.2 MaskFormerFusionHead, CGG's class-embedding scores) for the whole batch from
    the LOW-resolution logits.  probs (B, Q, C+1) class probabilities (column C = void); mask_pred_lowres (B, Q, h4, w4)
    fp32 or bf16.  Thresholds from test_cfg (default head.test_cfg): object_mask_thr 0.8, iou_thr 0.8, filter_low_score
    False.  Returns one (H_b, W_b) int32 map per image, each a view into one (B, Hmax, Wmax) buffer: label + 1000 *
    instance_id for things, label for stuff, C where no segment covers the pixel.  With stats=True also returns a dict of
    (B, Q) int32 tensors per query id: mask_area, original_area (0 for queries not kept) and seg_value (-1 where the
    query has no segment).  No host sync."""
    if not mask_pred_lowres.is_cuda:
        raise _lib.CggError('panoptic_postprocess_fused runs on CUDA only')
    cfg = dict(head.test_cfg or {}) if test_cfg is None else dict(test_cfg)
    rt, lib, h, s = _ctx(head, mask_pred_lowres.device)
    mp = mask_pred_lowres.contiguous()
    assert mp.dtype in (torch.float32, torch.bfloat16)
    B, Q, h4, w4 = mp.shape
    pr = probs.detach().float().contiguous()
    if tuple(pr.shape) != (B, Q, head.num_classes + 1):
        raise _lib.CggError('probs must be (B, Q, num_classes + 1) = %s, got %s' % ((B, Q, head.num_classes + 1),
                                                                                  tuple(pr.shape)))
    up = img_metas[0]['batch_input_shape']
    crops = [m['img_shape'][:2] for m in img_metas]
    outs = [m['ori_shape'][:2] for m in img_metas] if rescale else crops
    dev = mp.device
    geom = _geom([(c[0], c[1], o[0], o[1]) for c, o in zip(crops, outs)], dev)
    Hm, Wm = max(o[0] for o in outs), max(o[1] for o in outs)
    pan = torch.empty((B, Hm, Wm), dtype=torch.int32, device=dev)
    st = {k: torch.empty((B, Q), dtype=torch.int32, device=dev) for k in ('mask_area', 'original_area', 'seg_value')} \
        if stats else None
    nbytes = lib.cgg_panoptic_scratch_bytes(B, Q)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.cgg_panoptic_fuse(h, _p(mp), int(mp.dtype == torch.bfloat16), _p(pr), _p(geom), B, Q, pr.shape[-1],
                                     head.num_things_classes, h4, w4, up[0], up[1], Hm, Wm,
                                     float(cfg.get('object_mask_thr', 0.8)), float(cfg.get('iou_thr', 0.8)),
                                     int(bool(cfg.get('filter_low_score', False))), _p(pan),
                                     _p(st['mask_area']) if st else None, _p(st['original_area']) if st else None,
                                     _p(st['seg_value']) if st else None, _p(scratch), nbytes, s),
               h, 'cgg_panoptic_fuse')
    maps = [pan[b, :outs[b][0], :outs[b][1]] for b in range(B)]
    return (maps, st) if stats else maps


def class_probs(head, mask_cls_results, mask_cls_emb_results):
    """(B, Q, C+1) class probabilities of the fusion head: softmax(cls_emb @ class_embs^T) when the head uses class
    embeddings (get_cls_emb_scores), otherwise softmax(cls_logits) (mmdet's F.softmax(mask_cls, dim=-1))."""
    if head.use_class_emb:
        return cls_emb_scores(head, mask_cls_emb_results, head.class_embs)
    rt, lib, h, s = _ctx(head, mask_cls_results.device)
    x = mask_cls_results.detach().float().contiguous().clone()
    _lib.check(lib.cgg_softmax_rows(h, _p(x), x.numel() // x.shape[-1], x.shape[-1], s), h, 'cgg_softmax_rows')
    return x


def fusion_simple_test(head, mask_cls_results, mask_cls_emb_results, mask_pred_lowres, img_metas, rescale=False):
    """The fusion head's `simple_test` (maskformer_fusion_head.py:369-464) from the last head call's LOW-resolution mask
    logits (B, Q, h4, w4) instead of the upsampled ones.  Flags from head.test_cfg (mmdet's defaults: panoptic_on True,
    semantic_on False, instance_on False).  Returns one dict per image: 'pan_results' ((H, W) int32, see
    panoptic_postprocess_fused) when panoptic_on and 'ins_results' ((labels, bboxes, packed masks, (H, W)), see
    instance_postprocess_emb_fused) when instance_on."""
    cfg = dict(head.test_cfg or {})
    panoptic_on = cfg.get('panoptic_on', True)
    semantic_on = cfg.get('semantic_on', False)
    instance_on = cfg.get('instance_on', False)
    if semantic_on:
        raise NotImplementedError('semantic_postprocess is not implemented (as in mmdet 2.28.2)')
    B = mask_pred_lowres.shape[0]
    results = [dict() for _ in range(B)]
    if panoptic_on:
        probs = class_probs(head, mask_cls_results, mask_cls_emb_results)
        for r, m in zip(results, panoptic_postprocess_fused(head, probs, mask_pred_lowres, img_metas, rescale=rescale)):
            r['pan_results'] = m
    if instance_on:
        if not head.use_class_emb:
            raise _lib.CggError('instance results are built on the class embeddings (instance_postprocess_emb): '
                                'the head needs use_class_emb=True')
        ins = instance_postprocess_emb_fused(head, mask_cls_emb_results, mask_pred_lowres, head.class_embs, img_metas,
                                             rescale=rescale, max_per_image=cfg.get('max_per_image', 100))
        for r, x in zip(results, ins):
            r['ins_results'] = x
    return results
