"""CPU tests of the argument checks of the caption generator and its batched beam search (cgg_b200/caption.py): they
come before anything touches the device, so a malformed call fails the same way with or without a GPU."""
import pytest
import torch

from cgg_b200 import synth
from cgg_b200.lib import CggError
from cgg_b200.caption import CaptionTransformerB200, beam_search, beam_search_batch

CFG = synth.CAPTION_CFG_SMALL


class _Head:
    def __init__(self):
        self.caption_generator = CaptionTransformerB200(**CFG)


def test_forward_rejects_memory_and_tgt_of_different_batch():
    m = CaptionTransformerB200(**CFG)
    with pytest.raises(CggError, match='memory has 2 images, tgt 1'):
        m(torch.zeros((1, 3, 768)), torch.zeros((2, 12, 768)))


@pytest.mark.parametrize('kw', [dict(beam_width=0), dict(beam_width=33), dict(max_len=0), dict(max_len=36)])
def test_beam_search_rejects_out_of_range_arguments(kw):
    with pytest.raises(CggError):
        beam_search_batch(_Head(), torch.zeros((2, 12, 768)), **kw)


def test_beam_search_takes_one_image():
    with pytest.raises(CggError, match='one image'):
        beam_search(_Head(), torch.zeros((2, 12, 768)))
