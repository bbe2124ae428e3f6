"""CPU tests: the oracle (numpy + C) and the torch-op port against the golden vectors produced by the reference
module, and against each other."""
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, golden_names, load_golden
from oracle import c_oracle, cspn_numpy as onp


@pytest.mark.parametrize('name', golden_names())
def test_numpy_oracle_matches_reference_golden(name):
    c = load_golden(name)
    out = onp.cspn2d(c['guidance'], c['blur'], c['sparse_depth'], c['prop_time'], c['norm_type'])
    ok, ratio, normwise = onp.parity_ok(out, c['out'], rtol=1e-4)
    assert ok, (name, ratio, normwise)
    assert ratio < 0.05      # in practice the restatement is ~1e-7 normwise from the reference


@pytest.mark.parametrize('name', golden_names())
def test_c_oracle_matches_reference_golden(name):
    c = load_golden(name)
    out = c_oracle.cspn2d(c['guidance'], c['blur'], c['sparse_depth'], c['prop_time'], c['norm_type'])
    ok, ratio, normwise = onp.parity_ok(out, c['out'], rtol=1e-4)
    assert ok, (name, ratio, normwise)
    assert ratio < 0.05


def test_fp64_spec_bounds_fp32_rounding():
    c = load_golden('nyu_8sum')
    out64 = onp.cspn2d(c['guidance'], c['blur'], c['sparse_depth'], c['prop_time'], c['norm_type'], dtype=np.float64)
    ok, ratio, normwise = onp.parity_ok(c['out'], out64)
    assert ok and normwise < 1e-6


@pytest.mark.parametrize('norm', ['8sum', '8sum_abs'])
@pytest.mark.parametrize('shape', [(2, 3, 7, 9), (1, 1, 16, 33)])
def test_oracles_and_torch_port_match_live_reference(norm, shape):
    """tests/golden/port: inputs and the reference module's output, recorded by tests/golden/make_golden.py."""
    import torch
    from oracle import cspn_torch_port as tp
    z = np.load(os.path.join(GOLDEN_DIR, 'port', f'{norm}_' + 'x'.join(map(str, shape)) + '.npz'))
    g, d, s, ref = z['guidance'], z['blur'], z['sparse_depth'], z['out']
    assert g.shape == (shape[0], 9) + shape[2:] and d.shape == shape and str(z['norm_type']) == norm
    with torch.no_grad():
        port = tp.cspn2d_torch(torch.from_numpy(g), torch.from_numpy(d), torch.from_numpy(s), 6, norm).numpy()
    assert np.array_equal(port, ref)       # same op sequence -> same bits
    for out in (onp.cspn2d(g, d, s, 6, norm), c_oracle.cspn2d(g, d, s, 6, norm)):
        ok, ratio, _ = onp.parity_ok(out, ref)
        assert ok and ratio < 0.05


def test_semantics_pinned_by_reference():
    """Facts SURVEY.md 8(a) lists, checked on the oracle: sparse pixels return the BLUR depth
    (not the sparse value); prop_time=0 is the identity; extra guidance channels are ignored;
    '8sum_abs' has gate_sum == 1 in the interior."""
    rng = np.random.default_rng(0)
    g = rng.standard_normal((1, 10, 9, 11)).astype(np.float32)
    d = (rng.random((1, 1, 9, 11)) * 10).astype(np.float32)
    sp = np.zeros_like(d)
    sp[0, 0, 4, 5] = 3.0
    out = onp.cspn2d(g, d, sp, 5, '8sum')
    assert out[0, 0, 4, 5] == d[0, 0, 4, 5]
    assert np.array_equal(onp.cspn2d(g, d, sp, 0, '8sum'), d)
    assert np.array_equal(onp.cspn2d(g[:, :8], d, sp, 3, '8sum'), onp.cspn2d(g, d, sp, 3, '8sum'))
    _, gs = onp.affinity_normalization_2d(g, '8sum_abs')
    assert np.allclose(gs, 1.0, atol=1e-6)


@pytest.mark.parametrize('mode', ['26sum', '26sum_abs', 'paddle'])
def test_3d_c_oracle_matches_numpy(mode):
    rng = np.random.default_rng(1)
    g = rng.standard_normal((2, 26, 5, 6, 7)).astype(np.float32)
    f = rng.random((2, 2, 5, 6, 7)).astype(np.float32)
    a = onp.cspn3d(g, f, 4, mode)
    b = c_oracle.cspn3d(g, f, 4, mode)
    ok, ratio, _ = onp.parity_ok(b, a)
    assert ok and ratio < 0.05


def test_3d_reduces_to_2d_when_depth_is_one():
    """With D == 1 only the 8 in-plane channels (dz == 0) can contribute: the 3D definition must
    collapse onto the pinned 2D arithmetic (the only anchor the unpinned 3D path has)."""
    rng = np.random.default_rng(2)
    g3 = rng.standard_normal((1, 26, 1, 8, 9)).astype(np.float32)
    f = rng.random((1, 1, 1, 8, 9)).astype(np.float32)
    inplane = [k for k, o in enumerate(onp.OFFSETS_3D) if o[0] == 0]
    assert [onp.OFFSETS_3D[k][1:] for k in inplane] == list(onp.OFFSETS_2D)
    out3 = onp.cspn3d(g3, f, 5, '26sum')
    out2 = onp.cspn2d(g3[:, inplane, 0], f[:, :, 0], None, 5, '8sum')
    assert np.allclose(out3[:, :, 0], out2, rtol=1e-5, atol=1e-6)


def test_3d_paddle_mode_preserves_constants():
    """demo.py:47-49 normalises the gate to sum 1 at every voxel, so a constant volume is a fixed
    point in the interior (the property the Paddle op's documented contract implies)."""
    rng = np.random.default_rng(3)
    g = rng.random((1, 26, 6, 6, 6)).astype(np.float32) + 0.1
    f = np.full((1, 1, 6, 6, 6), 2.5, np.float32)
    out = onp.cspn3d(g, f, 1, 'paddle')
    assert np.allclose(out[0, 0, 1:-1, 1:-1, 1:-1], 2.5, rtol=1e-5)
