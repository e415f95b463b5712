"""Plain-torch restatement of the fusion head's panoptic output: mmdet 2.28.2 `MaskFormerFusionHead.panoptic_postprocess`
with the class-embedding probabilities in place of the class logits (the substitution CGG's `instance_postprocess_emb`
makes), after the resample chain of `Mask2FormerHeadOpen.simple_test` (bilinear upsample to batch_input_shape) and of
the fusion head's `simple_test` (crop to img_shape, optional bilinear resample to ori_shape).  Runs on CPU and GPU tensors;
the `sigmoid >= 0.5` cutoff is that of the device's sigmoid (CUDA: x > -1.7881392e-07), so comparisons with the CUDA
kernels run it on the GPU.

`hf_semantics=True` switches the two places where HuggingFace's independent implementation
(`transformers.models.mask2former.image_processing_mask2former.compute_segments`) differs from mmdet: HF counts
`original_area` on the score-scaled probabilities (it scales `mask_probs` in place before the loop) and drops a segment
when `ratio <= thr` where mmdet drops it when `ratio < thr`."""
import torch
import torch.nn.functional as F

INSTANCE_OFFSET = 1000


def resample_logits(mask_pred_lowres, batch_input_shape, img_shape, ori_shape=None):
    """(Q, h4, w4) low-resolution logits -> (Q, H, W) fp32: upsample to batch_input_shape, crop to img_shape and, when
    ori_shape is given (rescale), resample to it.  All bilinear with align_corners=False."""
    mp = F.interpolate(mask_pred_lowres.float()[None], size=tuple(batch_input_shape[:2]), mode='bilinear',
                       align_corners=False)[0]
    mp = mp[:, :img_shape[0], :img_shape[1]]
    if ori_shape is not None:
        mp = F.interpolate(mp[:, None], size=tuple(ori_shape[:2]), mode='bilinear', align_corners=False)[:, 0]
    return mp


def panoptic_postprocess(probs, mask_pred, num_things_classes, object_mask_thr=0.8, iou_thr=0.8, filter_low_score=False,
                         hf_semantics=False):
    """probs (Q, C+1) class probabilities (column C = void); mask_pred (Q, H, W) fp32 logits at the output size.
    Returns (pan (H, W) int32, stats) where stats holds, per query id, `mask_area`, `original_area` (0 for queries that
    were not kept) and `seg_value` (-1 where the query has no segment), plus `keep` and `prob_masks` (the kept queries'
    score * sigmoid, for margin computations)."""
    Q, C1 = probs.shape
    C = C1 - 1
    scores, labels = probs.max(-1)
    mask_pred = mask_pred.sigmoid()
    keep = labels.ne(C) & (scores > object_mask_thr)
    cur_scores, cur_classes, cur_masks = scores[keep], labels[keep], mask_pred[keep]
    cur_prob_masks = cur_scores.view(-1, 1, 1) * cur_masks
    h, w = cur_masks.shape[-2:]
    pan = torch.full((h, w), C, dtype=torch.int32, device=cur_masks.device)
    mask_area_q = torch.zeros(Q, dtype=torch.int64)
    original_area_q = torch.zeros(Q, dtype=torch.int64)
    seg_value_q = torch.full((Q,), -1, dtype=torch.int64)
    kept_ids = keep.nonzero()[:, 0].tolist()
    if cur_masks.shape[0] > 0:
        cur_mask_ids = cur_prob_masks.argmax(0)
        instance_id = 1
        for k in range(cur_classes.shape[0]):
            pred_class = int(cur_classes[k].item())
            isthing = pred_class < num_things_classes
            mask = cur_mask_ids == k
            mask_area = mask.sum().item()
            area_src = cur_prob_masks[k] if hf_semantics else cur_masks[k]
            original_area = (area_src >= 0.5).sum().item()
            mask_area_q[kept_ids[k]] = mask_area
            original_area_q[kept_ids[k]] = original_area
            if filter_low_score:
                mask = mask & (cur_masks[k] >= 0.5)
            if mask_area > 0 and original_area > 0:
                ratio = mask_area / original_area
                if (ratio <= iou_thr) if hf_semantics else (ratio < iou_thr):
                    continue
                if not isthing:
                    value = pred_class
                else:
                    value = pred_class + instance_id * INSTANCE_OFFSET
                    instance_id += 1
                pan[mask] = value
                seg_value_q[kept_ids[k]] = value
    return pan, dict(mask_area=mask_area_q, original_area=original_area_q, seg_value=seg_value_q, keep=keep,
                     prob_masks=cur_prob_masks)


def panoptic_from_lowres(probs, mask_pred_lowres, meta, num_things_classes, rescale=False, **kw):
    """One image: the resample chain, then panoptic_postprocess.  meta holds batch_input_shape, img_shape, ori_shape."""
    mp = resample_logits(mask_pred_lowres, meta['batch_input_shape'], meta['img_shape'],
                         meta['ori_shape'] if rescale else None)
    return panoptic_postprocess(probs, mp, num_things_classes, **kw)
