"""TEST INFRASTRUCTURE -- CPU restatement of the panoptic target preparation that feeds the matching-based losses:
mmdet 2.28.2 `MaskFormerHead.preprocess_gt` (mmdet/models/dense_heads/maskformer_head.py), which the reference calls at
open_set/models/mask2former_head.py:903, and the function it maps over the images, `preprocess_panoptic_gt`
(mmdet/core/utils/panoptic_gt_processing.py).  Only tests/ and tools/ import this file; the product
(betrayed-by-captions_b200/matching.py `preprocess_gt`) never does.

mmdet is not installed next to this tree, so the functions below are pinned on mmdet 2.28.2's source text, restated in
plain torch over dense tensors:

    things_masks = gt_masks.pad(img_metas['pad_shape'][:2], pad_val=0).to_tensor(dtype=torch.bool, device=...)
    if gt_semantic_seg is None:
        return gt_labels, things_masks.long()
    gt_semantic_seg = gt_semantic_seg.squeeze(0)
    semantic_labels = torch.unique(gt_semantic_seg, sorted=False, return_inverse=False, return_counts=False)
    for label in semantic_labels:
        if label < num_things or label >= num_things + num_stuff:
            continue
        stuff_masks_list.append(gt_semantic_seg == label); stuff_labels_list.append(label)
    labels = cat(things_labels, stack(stuff_labels)); masks = cat(things_masks, stack(stuff_masks)).long()

`torch.unique(..., sorted=False)` returns sorted values on a CUDA tensor, and the reference trains on CUDA, so the stuff
targets follow in ascending label order; that is what is restated here (tests/test_gpu_panoptic_targets.py pins the CUDA
behaviour).  `BitmapMasks.pad` puts the masks at the top-left of a zero plane of the padded size."""
import torch


def pad_masks(masks, pad_hw):
    """BitmapMasks.pad(pad_shape, pad_val=0): (G, h, w) -> (G, Hp, Wp), the masks at the top-left."""
    G, h, w = masks.shape
    out = masks.new_zeros((G,) + tuple(int(v) for v in pad_hw))
    out[:, :h, :w] = masks
    return out


def preprocess_panoptic_gt(gt_labels, gt_masks, gt_semantic_seg, num_things, num_stuff, img_metas):
    """One image: gt_labels (G,), gt_masks (G, h, w) (BitmapMasks.masks as a tensor), gt_semantic_seg (1, Hs, Ws) or None
    -> (labels (G + S,) int64, masks (G + S, Hp, Wp) int64).  torch.cat raises, as mmdet's does, when the padded things
    extent differs from the semantic map's and there is a stuff target."""
    num_classes = num_things + num_stuff
    things_masks = pad_masks(torch.as_tensor(gt_masks), img_metas['pad_shape'][:2]).bool()
    gt_labels = torch.as_tensor(gt_labels).long()
    if gt_semantic_seg is None:
        return gt_labels, things_masks.long()
    sem = torch.as_tensor(gt_semantic_seg).squeeze(0)
    stuff_masks, stuff_labels = [], []
    for label in torch.unique(sem, sorted=True):                # CUDA's order for sorted=False (module docstring)
        if label < num_things or label >= num_classes:
            continue
        stuff_masks.append(sem == label)
        stuff_labels.append(label)
    if stuff_masks:
        labels = torch.cat([gt_labels, torch.stack(stuff_labels, 0).long()], 0)
        masks = torch.cat([things_masks, torch.stack(stuff_masks, 0)], 0)
    else:
        labels, masks = gt_labels, things_masks
    return labels, masks.long()


def preprocess_gt(gt_labels_list, gt_masks_list, gt_semantic_segs, img_metas, num_things, num_stuff):
    """MaskFormerHead.preprocess_gt: preprocess_panoptic_gt over the images -> (labels_list, masks_list)."""
    if gt_semantic_segs is None:
        gt_semantic_segs = [None] * len(gt_labels_list)
    out = [preprocess_panoptic_gt(l, m, s, num_things, num_stuff, meta)
           for l, m, s, meta in zip(gt_labels_list, gt_masks_list, gt_semantic_segs, img_metas)]
    return [o[0] for o in out], [o[1] for o in out]
