"""CPU-only checks of the C-ABI boundary: the library builds, loads, and exports every symbol
that include/gen6d_b200.h declares; the ctypes binding covers all of them; the product path
fails loudly without a GPU (no fallback)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from gen6d_b200 import _lib


@pytest.fixture(scope='module')
def built():
    from gen6d_b200.build import build
    return build()


def test_library_exports_every_declared_symbol(built):
    lib = ctypes.CDLL(built)
    names = _lib.header_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f'{n} declared in include/gen6d_b200.h but not exported'


def test_binding_covers_header(built):
    bound = set(_lib._SIGNATURES) | {'g6d_last_error', 'g6d_version', 'g6d_launch_count'}
    assert set(_lib.header_symbols()) == bound


def test_error_reporting_without_gpu(built):
    l = _lib.lib()
    assert l.g6d_version() >= 100
    d = _lib.ConvDesc()  # all zeros -> invalid
    assert l.g6d_conv_workspace_bytes(ctypes.byref(d)) == -1
    assert b'bad dims' in l.g6d_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the no-GPU failure mode')
def test_compute_fails_loudly_without_cuda():
    from gen6d_b200.network import name2network
    det = name2network['detector']({})
    with pytest.raises(Exception):
        det.load_ref_imgs(np.zeros((2, 128, 128, 3), np.uint8))


def _bench_module():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('g6d_bench', os.path.join(root, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_batch_choice_deals_lanes_evenly():
    """bench.py's pick_batch: the timed region of `steps` poses is dealt to the lanes as equal numbers of full batches
    whenever the step count allows it (the default 20 steps on 2 lanes -> 2 x 10)."""
    bench = _bench_module()
    if bench.E2E_BATCH > 0:
        pytest.skip('G6D_E2E_BATCH overrides the choice')
    want = {(20, 2): 10, (16, 2): 8, (24, 2): 6, (14, 2): 7, (20, 1): 10, (4, 2): 2, (2, 2): 1, (22, 2): 4, (5, 2): 1,
            (9, 2): 4, (40, 2): 10, (30, 3): 10}
    for (steps, lanes), b in want.items():
        assert bench.pick_batch(steps, lanes) == b, (steps, lanes)
        if steps % lanes == 0 and (steps // lanes) % b == 0:
            assert (steps // b) % lanes == 0          # every lane runs the same number of batches


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: stage outputs named by stage and output, float32 / float64 only, integers exact, an
    oversized array replaced by the same seeded sample on every run, and the whole dump within the byte limit."""
    bench = _bench_module()
    chain = torch.arange(24, dtype=torch.float64).reshape(2, 1, 3, 4)
    idx = torch.tensor([3, 2**31 - 1], dtype=torch.int32)
    crop = torch.arange(2 * 64 * 64 * 3, dtype=torch.int32).reshape(2, 64, 64, 3).to(torch.uint8)
    outs = [('predict', (chain, torch.zeros(2, 4), crop, idx, torch.ones(2, 3), torch.ones(2, 5, dtype=torch.float16))),
            ('refine', torch.ones(2, 6)), ('refine', torch.zeros(2, 6))]
    arrays = bench.stage_outputs(outs)
    assert sorted(arrays) == ['predict.crop', 'predict.detection', 'predict.logits', 'predict.poses', 'predict.ref_idx',
                              'predict.selection', 'refine0.0', 'refine1.0']
    limit = 64 << 10
    for d in ('a', 'b'):
        written = bench.write_outputs(str(tmp_path / d), arrays, limit)
        assert written['predict.crop'][1] == [2, 64, 64, 3] and written['predict.crop'][0][0] < crop.numel()
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= limit
    for name in arrays:
        a, b = np.load(tmp_path / 'a' / f'{name}.npy'), np.load(tmp_path / 'b' / f'{name}.npy')
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.testing.assert_array_equal(a, b)
    assert np.load(tmp_path / 'a' / 'predict.poses.npy').dtype == np.float64
    np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'predict.poses.npy'), chain.numpy())
    np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'predict.ref_idx.npy'), [3, 2**31 - 1])
    crop_s = np.load(tmp_path / 'a' / 'predict.crop.npy')
    assert set(crop_s.astype(np.int64)) <= set(crop.numpy().reshape(-1).astype(np.int64))
