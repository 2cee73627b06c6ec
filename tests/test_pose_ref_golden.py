"""The two-view pose oracle is PINNED: tests/golden/pose_*.npz were produced by the reference's own
``pose_optimization/two_view/*.py`` (imported unmodified through oracle/ref_shim.py by
oracle/make_pose_golden.py).  Here oracle/pose.py is re-checked against those files on any box (CPU)."""
import glob
import json
import os

import numpy as np
import pytest

from tests.util import GOLDEN

W8PT = sorted(glob.glob(os.path.join(GOLDEN, 'pose_w8pt_n*.npz')))
BA = sorted(glob.glob(os.path.join(GOLDEN, 'pose_ba_*.npz')))


def tdir(T):
    t = T[..., :3, 3]
    return t / np.linalg.norm(t, axis=-1, keepdims=True)


def test_fixture_inventory():
    assert len(W8PT) >= 8 and len(BA) >= 7
    rep = json.load(open(os.path.join(GOLDEN, 'pose_report.json')))
    # the generator asserted oracle == reference; the report keeps the measured deviations
    assert max(v for k, v in rep.items() if k.endswith('64_oracle_err')) < 1e-8
    assert all(v == 0 for k, v in rep.items() if 'mask_flips' in k)


@pytest.mark.parametrize('path', W8PT, ids=[os.path.basename(p)[5:-4] for p in W8PT])
def test_w8pt_oracle_vs_reference_golden(path):
    from oracle import pose as P
    z = np.load(path)
    for tag, dt, tol in (('64', np.float64, 1e-9), ('32', np.float32, 2e-5)):
        T, info = P.estimate_relative_pose_w8pt(z['kpts0'].astype(dt), z['kpts1'].astype(dt), z['intr'].astype(dt),
                                                z['intr'].astype(dt), z['conf'].astype(dt), determine_inliers=True)
        assert np.abs(T - z['T' + tag]).max() < tol
        if dt == np.float64:
            assert np.array_equal(info['pos_depth_mask'], z['pos64'])
            assert np.array_equal(info['inliers'], z['inl64'])
            np.testing.assert_allclose(info['confidence'], z['conf64'], rtol=1e-12)
            np.testing.assert_allclose(info['kpts0_norm'], z['k0n64'], atol=1e-12)


def test_w8pt_choose_closest_oracle_vs_reference_golden():
    from oracle import pose as P
    z = np.load(os.path.join(GOLDEN, 'pose_w8pt_closest_b4_n200.npz'))
    T, info = P.estimate_relative_pose_w8pt(*(z[k].astype(np.float64) for k in ('kpts0', 'kpts1', 'intr', 'intr', 'conf')),
                                            choose_closest=True, T_021=z['T_gt'].astype(np.float64))
    assert np.abs(T - z['T64']).max() < 1e-9
    assert np.array_equal(info['pos_depth_mask'], z['pos64'])


@pytest.mark.parametrize('path', BA, ids=[os.path.basename(p)[5:-4] for p in BA])
def test_ba2view_oracle_vs_reference_golden(path):
    from oracle import pose as P
    z = np.load(path)
    ext, valid = P.run_bundle_adjust_2_view(z['kpts0_norm'].astype(np.float64), z['kpts1_norm'].astype(np.float64),
                                            z['conf'].astype(np.float64), z['T_init'].astype(np.float64), 10)
    assert np.array_equal(valid, z['valid64']) and np.array_equal(valid, z['valid32'])
    if ext.size:
        assert np.abs(ext - z['ext64']).max() < 1e-7
