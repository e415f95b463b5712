"""CPU tests of the panoptic training targets: the oracle's restatement of mmdet 2.28.2 `preprocess_gt`
(oracle/panoptic_targets_oracle.py) against hand-built expectations, and the host-side checks of the product's
`preprocess_gt` (cgg_b200/matching.py), which reject bad input before any device work."""
import numpy as np
import pytest
import torch

from oracle import panoptic_targets_oracle as PT
from cgg_b200 import matching
from cgg_b200.lib import CggError

NT, NS = 4, 3                      # things 0..3, stuff 4..6; 7+ and 255 are no class


class Bitmap:
    """The part of mmdet's BitmapMasks that preprocess_gt reads."""

    def __init__(self, masks):
        self.masks = np.asarray(masks, dtype=np.uint8)
        self.height, self.width = self.masks.shape[1:]


def _meta(h, w):
    return dict(pad_shape=(h, w, 3))


def test_things_only_are_padded_at_the_top_left():
    m = torch.zeros((2, 3, 4), dtype=torch.uint8)
    m[0, 0, 0] = m[1, 2, 3] = 1
    labels, masks = PT.preprocess_gt([torch.tensor([2, 0])], [m], None, [_meta(5, 6)], NT, NS)
    assert labels[0].tolist() == [2, 0] and masks[0].dtype == torch.int64 and masks[0].shape == (2, 5, 6)
    want = torch.zeros((2, 5, 6), dtype=torch.long)
    want[0, 0, 0] = want[1, 2, 3] = 1
    assert torch.equal(masks[0], want)


def test_things_then_stuff_in_ascending_order_other_values_ignored():
    sem = torch.full((1, 4, 4), 255, dtype=torch.uint8)
    sem[0, 0] = torch.tensor([6, 6, 1, 9])            # 6 stuff, 1 a thing label, 9 >= num_classes
    sem[0, 1] = torch.tensor([4, 4, 7, 255])          # 4 stuff, 7 == num_classes
    m = torch.ones((1, 2, 2), dtype=torch.bool)
    labels, masks = PT.preprocess_gt([torch.tensor([3])], [m], sem.unsqueeze(0), [_meta(4, 4)], NT, NS)
    assert labels[0].tolist() == [3, 4, 6]
    assert masks[0].shape == (3, 4, 4)
    assert masks[0][1].nonzero().tolist() == [[1, 0], [1, 1]]
    assert masks[0][2].nonzero().tolist() == [[0, 0], [0, 1]]
    assert int(masks[0][0].sum()) == 4


def test_stuff_only_empty_image_and_a_single_corner_pixel():
    sem = torch.full((1, 3, 5), 255, dtype=torch.int64)
    sem[0, 2, 4] = 5                                   # one corner pixel
    empty = torch.zeros((0, 3, 5), dtype=torch.uint8)
    labels, masks = PT.preprocess_gt([torch.zeros((0,), dtype=torch.long)] * 2, [empty, empty],
                                     torch.stack([sem, torch.full((1, 3, 5), 255)]), [_meta(3, 5)] * 2, NT, NS)
    assert labels[0].tolist() == [5] and masks[0][0].nonzero().tolist() == [[2, 4]]
    assert labels[1].tolist() == [] and masks[1].shape == (0, 3, 5)


def test_every_stuff_class_ascending_whatever_the_pixel_order():
    sem = torch.tensor([[[6, 5, 4, 2]]], dtype=torch.uint8)
    labels, _ = PT.preprocess_gt([torch.tensor([0])], [torch.ones((1, 1, 4), dtype=torch.uint8)], [sem], [_meta(1, 4)], NT, NS)
    assert labels[0].tolist() == [0, 4, 5, 6]


def test_oracle_concatenation_fails_on_a_shape_mismatch_with_stuff_only():
    m = torch.ones((1, 2, 2), dtype=torch.uint8)
    no_stuff = torch.full((1, 1, 3, 3), 255, dtype=torch.uint8)
    PT.preprocess_gt([torch.tensor([0])], [m], no_stuff, [_meta(4, 4)], NT, NS)
    with pytest.raises(RuntimeError):
        PT.preprocess_gt([torch.tensor([0])], [m], torch.full((1, 1, 3, 3), 5, dtype=torch.uint8), [_meta(4, 4)], NT, NS)


def test_stuff_extent_check_raises_only_with_stuff_targets():
    metas = [_meta(4, 4), _meta(3, 3)]
    matching.check_stuff_extent([0, 2], metas, (3, 3))
    matching.check_stuff_extent([0, 0], metas, (5, 5))
    with pytest.raises(CggError):
        matching.check_stuff_extent([1, 0], metas, (3, 3))


def test_preprocess_gt_rejects_bad_input_on_the_host():
    sem = torch.full((1, 1, 4, 4), 255, dtype=torch.uint8)
    with pytest.raises(CggError, match='2 masks for 1 labels'):
        matching.preprocess_gt([torch.tensor([0])], [Bitmap(np.ones((2, 4, 4)))], sem, [_meta(4, 4)], NT, NS, 'cuda')
    with pytest.raises(CggError, match='uint8 or int64'):
        matching.preprocess_gt([torch.tensor([0])], [Bitmap(np.ones((1, 4, 4)))], sem.int(), [_meta(4, 4)], NT, NS, 'cuda')
    with pytest.raises(CggError, match='larger than pad_shape'):
        matching.preprocess_gt([torch.tensor([0])], [Bitmap(np.ones((1, 5, 4)))], None, [_meta(4, 4)], NT, NS, 'cuda')
    with pytest.raises(CggError, match='bool or uint8'):
        matching.preprocess_gt([torch.tensor([0])], [torch.ones((1, 4, 4))], None, [_meta(4, 4)], NT, NS, 'cuda')
