"""GPU tests of the batched caption beam search (cgg_b200/caption.py `beam_search_batch`, csrc/caption_kernels.cu): for
every image of a batch, the result of the oracle's beam search (oracle/caption_oracle.py, pinned on the live reference)
run on that image alone on the CPU -- the same finished sequences in the same order, the same best sentence, scores
within 1e-4 relative.  Every case is checked to have no exact tie among the W + 1 best candidates of any selection, so
that the sequences are decided by the arithmetic and not by a tie-break."""
import contextlib

import pytest
import torch

from oracle import caption_oracle as CO
from cgg_b200 import synth
from cgg_b200 import lib as _lib
from cgg_b200.head import Mask2FormerHeadOpenB200
from cgg_b200.caption import beam_search, beam_search_batch, _search_device, _search_results
from test_caption_cpu import CFG, BOS, EOS

pytestmark = pytest.mark.gpu
DEV = 'cuda'
CFG_REAL = dict(nb_layers=4, input_dim=768, hidden_dim=768, ff_dim=512, nb_heads=8, drop_val=0.0, pre_norm=False,
                seq_length=35, nb_tokens=30522)


def _head(seed, cfg=CFG, eos_bias=2.0):
    sd = synth.make_caption_params(seed, cfg=cfg, eos_bias=eos_bias)
    head = Mask2FormerHeadOpenB200(num_things_classes=48, num_stuff_classes=0, num_queries=12, use_class_emb=True,
                                   use_caption=True, use_caption_generation=True, bert_vocab_size=cfg['nb_tokens'],
                                   caption_generator=dict(type='CaptionTransformer', **cfg))
    head.load_state_dict(sd, strict=False)
    sd['caption_generator.position_encoder.psne_layer'] = CO.positions(35, 768)
    return head.to(DEV).eval(), sd


@contextlib.contextmanager
def _topk_calls():
    """Records the input and picks of every torch.topk call (the oracle's selections)."""
    calls, orig = [], torch.topk

    def topk(x, k, **kw):
        v, i = orig(x, k, **kw)
        calls.append((x.flatten(), k, i))
        return v, i
    torch.topk = topk
    try:
        yield calls
    finally:
        torch.topk = orig


def _oracle(sd, cfg, memory, max_len=35, beam_width=7):
    """Per image: (best ids, finished, number of passes after the BOS step, topk picks of each selection)."""
    out = []
    for b in range(memory.shape[0]):
        with _topk_calls() as calls:
            best, finished = CO.beam_search(sd, cfg, memory[b:b + 1], BOS, EOS, max_len=max_len, beam_width=beam_width)
        for x, k, _ in calls:
            top = x.sort(descending=True).values[:k + 1]
            assert bool((top[:-1] > top[1:]).all()), 'exact tie at a selection boundary'
        out.append((best, finished, len(calls) - 1, [i for _, _, i in calls]))
    return out


def _assert_same(res, want):
    best, finished = want[0], want[1]
    assert [f[0] for f in res['finished']] == [f[0] for f in finished]
    assert res['ids'] == best
    for a, b in zip(res['finished'], finished):
        assert abs(a[1] - b[1]) <= 1e-4 * abs(b[1])
    if finished:
        assert res['score'] == res['finished'][[f[0] for f in res['finished']].index(best)][1]


def _memory(seed, B, Q=12):
    return torch.randn((B, Q, 768), generator=torch.Generator().manual_seed(seed))


def test_batch_of_images_finishing_at_different_passes():
    head, sd = _head(5, eos_bias=3.0)
    memory = _memory(11, 8)
    want = _oracle(sd, CFG, memory)
    assert len({w[2] for w in want}) > 1                      # the images end at different passes
    got = beam_search_batch(head, memory.to(DEV))
    assert len(got) == 8
    for res, w in zip(got, want):
        _assert_same(res, w)


def _stops_mid_list(want, beam_width):
    """The last pass's walk stopped at the beam_width-th finished sentence before its last pick."""
    best, finished, _, picks = want
    if len(finished) != beam_width:
        return False
    last_len = len(finished[-1][0])
    appended = sum(len(f[0]) == last_len for f in finished)
    eos_ranks = [r for r, p in enumerate(picks[-1].tolist()) if p % CFG['nb_tokens'] == EOS]
    return eos_ranks[appended - 1] < beam_width - 1


@pytest.mark.parametrize('case', ['stop_mid_list', 'nothing_finishes', 'max_len_6', 'beam_width_1', 'beam_width_3'])
def test_edge_cases(case):
    kw = dict(max_len=35, beam_width=7)
    eos_bias = 2.0
    if case == 'stop_mid_list':
        eos_bias = 6.0
    elif case == 'nothing_finishes':
        eos_bias = -50.0
    elif case == 'max_len_6':
        kw['max_len'] = 6
    else:
        kw['beam_width'] = int(case[-1])
    head, sd = _head(7, eos_bias=eos_bias)
    memory = _memory(13, 3)
    want = _oracle(sd, CFG, memory, **kw)
    got = beam_search_batch(head, memory.to(DEV), **kw)
    for res, w in zip(got, want):
        _assert_same(res, w)
    if case == 'stop_mid_list':
        assert any(_stops_mid_list(w, 7) for w in want)
    elif case == 'nothing_finishes':
        assert all(r['ids'] is None and r['finished'] == [] for r in got)
    elif case == 'max_len_6':                                 # beams are dropped: every sentence is shorter than max_len
        assert all(len(f[0]) <= 5 for r in got for f in r['finished'])
        assert any(w[2] == 3 for w in want)                   # a search that ran until no beam could continue


def test_real_config_batch_of_two():
    head, sd = _head(3, cfg=CFG_REAL)
    memory = _memory(17, 2, Q=100)
    want = _oracle(sd, CFG_REAL, memory)
    got = beam_search_batch(head, memory.to(DEV))
    for res, w in zip(got, want):
        _assert_same(res, w)


def test_simple_test_with_caption_batch_of_three():
    from test_gpu_post import _StubPixelDecoder
    Q, B = 12, 3
    sdh = synth.make_params(seed=6, num_queries=Q, perturb=True)
    sdc = synth.make_caption_params(5)
    head = Mask2FormerHeadOpenB200(num_things_classes=48, num_stuff_classes=0, num_queries=Q, use_class_emb=True,
                                   use_caption=True, use_caption_generation=True, bert_vocab_size=CFG['nb_tokens'],
                                   caption_generator=dict(type='CaptionTransformer', **CFG), pixel_decoder=_StubPixelDecoder())
    head.load_state_dict({**sdh, **sdc}, strict=False)
    head = head.to(DEV).eval()
    mf, mems = synth.make_inputs(8, B, 96, 128)
    feats = [mf.to(DEV)] + [m.to(DEV) for m in mems]
    with torch.no_grad():
        out = head.simple_test(feats, [dict(batch_input_shape=(96, 128))] * B, with_caption=True)
    assert isinstance(out[3], list) and len(out[3]) == B
    sdc['caption_generator.position_encoder.psne_layer'] = CO.positions(35, 768)
    want = _oracle(sdc, CFG, out[1].float().cpu())            # independent of the device search
    for b in range(B):
        assert out[3][b] == beam_search(head, out[1][b:b + 1].float())['ids']
        assert out[3][b] == want[b][0]


def test_no_blocking_sync_before_the_final_gather():
    head, _ = _head(5)
    memory = _memory(11, 4).to(DEV)
    want = beam_search_batch(head, memory)                    # warm-up: runtime, workspaces, module loads
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        st, steps = _search_device(head, memory, BOS, EOS, 35, 7, 0.7)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert 2 <= steps <= 33
    assert _search_results(st) == want


def test_out_of_range_arguments():
    head, _ = _head(5)
    memory = _memory(11, 2).to(DEV)
    for kw in (dict(beam_width=0), dict(beam_width=33), dict(max_len=36)):
        with pytest.raises(_lib.CggError):
            beam_search_batch(head, memory, **kw)
    # the C ABI's own checks: beam_width outside 1..32, max_len past the position table, non-positive sizes
    rt = head._runtime(torch.device(DEV))
    z = torch.zeros(64, dtype=torch.int64, device=DEV)
    st = _lib.BeamState(token_cap=8, **{n: z.data_ptr() for n in ('tokens', 'weights', 'n_active', 'parent', 'next_ids',
                                                                  'fin_tokens', 'fin_len', 'fin_score', 'n_fin', 'max_idx',
                                                                  'done', 'n_done')})
    p = z.data_ptr()
    sel = lambda batch, W, max_len, npos: rt.lib.cgg_caption_beam_select(                            # noqa: E731
        rt.handle, p, p, batch, W, 0, 2, max_len, npos, 1.0, 1.0, EOS, st, None)
    bad = -1                                                 # CGG_ERR_BAD_SHAPE
    assert sel(1, 33, 35, 35) == bad and sel(1, 0, 35, 35) == bad and sel(1, 7, 36, 35) == bad and sel(0, 7, 35, 35) == bad
    assert rt.lib.cgg_caption_beam_scores(rt.handle, p, 4, 1, 33, 100, 0, st, 1.0, p, p, None) == bad
    assert rt.lib.cgg_caption_self_attn_step(rt.handle, p, p, p, p, 0, 8, 96, 0, 4, 1.0, None) == bad
    assert rt.lib.cgg_caption_cache_reorder(rt.handle, p, p, p, 4, 1, 33, 4, 1, 768, None) == bad
    st.token_cap = 12032 // 7 + 1                            # the select kernel's token staging past its shared memory
    assert sel(1, 7, 35, 35) == bad
