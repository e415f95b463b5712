"""CPU-side checks: the C-ABI library builds/loads and exports every symbol declared in
include/cgg_b200.h; the host-side head mirrors the reference's state_dict layout; the product
path refuses to run without CUDA (no fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

from cgg_b200 import build as cbuild
from cgg_b200 import lib as clib
from cgg_b200 import synth
from cgg_b200.head import Mask2FormerHeadOpenB200

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    cbuild.build()
    return clib.load()


def test_library_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, 'include', 'cgg_b200.h')).read()
    declared = set(re.findall(r'\b(cgg_[a-z_0-9]+)\s*\(', hdr))
    declared -= {'cgg_handle'}
    assert len(declared) >= 16
    for name in sorted(declared):
        assert hasattr(lib, name), 'library does not export ' + name
    assert set(clib.EXPORTS) == declared


def test_version_names_sm100a(lib):
    assert b'sm_100a' in lib.cgg_version()


def test_sass_is_sm100a_only():
    import subprocess
    out = subprocess.run(['cuobjdump', '-lelf', clib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r'sm_(\d+a?)', out))
    assert archs == {'100a'}, archs


def test_sass_uses_blackwell_tensor_and_tma_paths():
    """The library's SASS carries tcgen05 MMAs (single-CTA and CTA-pair), TMEM loads, TMA loads and stores."""
    import subprocess
    sass = subprocess.run(['cuobjdump', '-sass', clib.LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ('UTCHMMA', 'UTCHMMA.2CTA', 'UTCBAR.2CTA.MULTICAST', 'LDTM', 'UTMALDG.3D', 'UTMALDG.2D.2CTA', 'UTMASTG.3D'):
        assert mnemonic in sass, mnemonic
    assert 'HMMA.16816' not in sass and 'WGMMA' not in sass      # no mma.sync / wgmma fallbacks


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the no-GPU behaviour')
def test_no_cpu_fallback(lib):
    h = C.c_void_p()
    cfg = clib.Config(100, 256, 8, 2048, 9, 49, 768, 0, 0)
    assert lib.cgg_create(C.byref(h), C.byref(cfg)) == -3      # CGG_ERR_CUDA
    head = Mask2FormerHeadOpenB200(num_things_classes=48, num_stuff_classes=0, num_queries=8)
    mf, mems = synth.make_inputs(0, 1, 64, 64)
    with pytest.raises(clib.CggError):
        head.decoder_forward(mf, mems)


def test_create_rejects_bad_config(lib):
    h = C.c_void_p()
    assert lib.cgg_create(C.byref(h), C.byref(clib.Config(100, 128, 8, 2048, 9, 49, 768, 0, 0))) == -2
    assert lib.cgg_create(C.byref(h), C.byref(clib.Config(100, 256, 8, 2048, 99, 49, 768, 0, 0))) == -1
    assert lib.cgg_create(None, None) == -6


def test_state_dict_keys_match_reference_layout():
    """SURVEY.md section 8b: the replacement must accept the reference's keys unchanged."""
    head = Mask2FormerHeadOpenB200(num_things_classes=48, num_stuff_classes=0, num_queries=100, use_class_emb=True)
    sd = synth.make_params(seed=0, num_queries=100, num_classes_p1=49)
    assert set(head.state_dict().keys()) == set(sd.keys())
    for k, v in head.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    n = sum(p.numel() for p in head.parameters())
    assert n == 14668593          # head-only parameter count of the reference (SURVEY.md 8b)
    head.load_state_dict(sd, strict=True)


def test_use_class_emb_false_has_no_v2l_transform():
    """head.py:178,202-219: the reference default builds neither v2l_transform nor class_embs (the class-agnostic
    pre-training configs); a checkpoint of such a model must load strictly."""
    head = Mask2FormerHeadOpenB200(num_things_classes=48, num_stuff_classes=0, num_queries=100, pred_emb_norm=True)
    keys = set(head.state_dict().keys())
    assert not any(k.startswith('v2l_transform') or k == 'class_embs' for k in keys)
    sd = {k: v for k, v in synth.make_params(seed=0, num_queries=100).items()
          if not k.startswith('v2l_transform') and k != 'class_embs'}
    head.load_state_dict(sd, strict=True)


def test_synth_is_deterministic():
    a = synth.make_params(seed=5, num_queries=12)
    b = synth.make_params(seed=5, num_queries=12)
    assert all(torch.equal(a[k], b[k]) for k in a)
    x, _ = synth.make_inputs(1, 1, 64, 96)
    y, _ = synth.make_inputs(1, 1, 64, 96)
    assert torch.equal(x, y) and x.shape == (1, 256, 16, 24)
    assert synth.level_sizes(1024, 1024) == ((256, 256), [(32, 32), (64, 64), (128, 128)])


def test_no_gc_during_capture_context():
    """CUDA-graph captures run with the cyclic collector off (a dropped head's cgg_destroy in the middle of a capture
    invalidates it) and the collector's state is restored afterwards."""
    import gc
    was = gc.isenabled()
    with clib.no_gc_during_capture():
        assert not gc.isenabled()
    assert gc.isenabled() == was
    gc.disable()
    try:
        with clib.no_gc_during_capture():
            assert not gc.isenabled()
        assert not gc.isenabled()          # it was off before: stays off
    finally:
        if was:
            gc.enable()


def test_bench_dump_outputs_fixed_sample_within_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: small arrays whole (shape kept), larger ones as one element from each of `cap` blocks
    that cover the array to its last element, at the same positions on every call, float32, within the byte budget."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, 'DUMP_BYTES', 3 * 4 * 1000)
    g = torch.Generator().manual_seed(0)
    outs = ([torch.randn((2, 5, 7), generator=g) for _ in range(10)], [torch.randn((1, 1, 199), generator=g) for _ in range(10)],
            [None] * 9 + [torch.randn((2, 5, 16, 16), generator=g).bfloat16()])
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), outs)
    got = {n: np.load(tmp_path / 'a' / (n + '.npy')) for n in ('cls', 'emb', 'mask')}
    assert all(v.dtype == np.float32 and np.array_equal(v, np.load(tmp_path / 'b' / (n + '.npy'))) for n, v in got.items())
    assert np.array_equal(got['cls'], torch.stack(outs[0]).numpy())
    # emb: 1990 elements, just under twice the 1000-element share: the blocks must still reach its last element
    for name, full in (('emb', torch.stack(outs[1])), ('mask', outs[2][-1].float())):
        full = full.reshape(-1).numpy()
        starts = [i * full.size // 1000 for i in range(1001)]
        assert got[name].shape == (1000,) and starts[-1] == full.size
        assert all(got[name][i] in full[starts[i]:starts[i + 1]] for i in range(1000)), name
        assert not np.array_equal(got[name], full[starts[:-1]])     # offsets within the blocks vary
    assert sum(f.stat().st_size for f in (tmp_path / 'a').iterdir()) <= bench.DUMP_BYTES + 3 * 128
