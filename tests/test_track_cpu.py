"""Pose smoothing of the video tracker (csrc/pnp_math.cuh, g6d_track_smooth) through its *_host twin -- the same
__host__ __device__ code the kernel runs -- against the numpy / OpenCV restatement of predict.py's smoothing
(oracle/track.py) and against the golden run of the unmodified reference's tracking loop.  CPU-only."""
import os

import cv2
import numpy as np
import pytest

from gen6d_b200 import glue
from oracle import track as T

HERE = os.path.dirname(os.path.abspath(__file__))
BBOX = T.bbox_corners(np.array([0.9, 0.7, 1.1]), np.array([-0.8, -0.6, -1.0])).astype(np.float32)


def ulps(a, b):
    """|a - b| in float32 ulps of b."""
    return float((np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.spacing(np.abs(b).astype(np.float32))).max())


def noisy_track(rng, n, f, px):
    """n float32 poses along a smooth path, jittered so that the corners move by up to ~px pixels from frame to frame
    (the weighted average of the history is then 0 - 2 px away from any single pose's projection)."""
    r0, z = rng.randn(3), 6 + rng.rand() * 4
    t0 = np.array([rng.randn() * 0.4, rng.randn() * 0.4, z])
    dr, dt = rng.randn(3) * 0.01, rng.randn(3) * 0.02
    out = []
    for k in range(n):
        jr = rng.randn(3) * px / f / 1.2 * rng.rand()
        jt = rng.randn(3) * px * z / f * rng.rand() * np.array([1, 1, z])
        R = cv2.Rodrigues(r0 + dr * k + jr)[0]
        out.append(np.concatenate([R, (t0 + dt * k + jt)[:, None]], 1).astype(np.float32))
    return out


def special_track(n, kind):
    """A box with one corner at |depth| < 1e-4 (project_points' clamp) or behind the camera."""
    R = cv2.Rodrigues(np.array([0.3, -0.2, 0.1]))[0].astype(np.float32)
    z0 = float((R @ BBOX[0].astype(np.float64))[2])
    tz = -z0 + (5e-5 if kind == 'clamp' else -0.4)
    return [np.concatenate([R, np.array([[0.05 * k], [0.02], [tz]])], 1).astype(np.float32) for k in range(n)]


def run_lanes(tracks, Ks, num, std):
    """Feed M lanes frame by frame through the host twin and the oracle; yields per (frame, lane) both results."""
    M, n = len(tracks), len(tracks[0])
    w, ws = glue.smoothing_weights(num, std)
    hist, cnt = np.zeros((M, num, 8, 2), np.float32), np.zeros(M, np.int32)
    cams = glue.cameras(np.stack(Ks))
    refs = [T.smooth_sequence(BBOX, tracks[l], Ks[l], num, std) for l in range(M)]
    for k in range(n):
        c, wp, sm = glue.host_track_smooth(BBOX, np.stack([t[k] for t in tracks]).astype(np.float64), cams, w, ws, hist, cnt)
        assert cnt.tolist() == [k + 1] * M
        for l in range(M):
            yield k, l, (c[l], wp[l], sm[l]), refs[l][k]


@pytest.mark.parametrize('num,std', [(5, 2.5), (10, 10.0)])
def test_host_twin_matches_opencv(num, std):
    """>= 100 seeded cases per (num, std): histories of length 1 ... num + 3 (the ring wraps), 0 - 2 px averaging noise,
    twelve lanes with their own intrinsics, plus a lane whose box touches the depth clamp and one with a corner behind the
    camera."""
    rng = np.random.RandomState(num)
    L = 12
    Ks = [np.array([[f, 0, 320], [0, f, 240], [0, 0, 1]], np.float32) for f in 500 + 400 * rng.rand(L)]
    tracks = [noisy_track(rng, num + 3, float(Ks[l][0, 0]), 25.0) for l in range(L)]
    tracks += [special_track(num + 3, 'clamp'), special_track(num + 3, 'behind')]
    Ks += [Ks[0], Ks[0]]
    worst = {'corners_ulp': 0., 'dR': 0., 'dt': 0., 'rms_px': 0.}
    cases = 0
    for k, l, (c, wp, sm), (c_ref, w_ref, p_ref) in run_lanes(tracks, Ks, num, std):
        assert ulps(c, c_ref) <= 2, (k, l)
        np.testing.assert_allclose(wp, w_ref, rtol=1e-15, atol=0)
        rms, rms_cv = T.reprojection_rms(BBOX, w_ref, sm, Ks[l]), T.reprojection_rms(BBOX, w_ref, p_ref, Ks[l])
        assert rms <= rms_cv * (1 + 1e-12) + 1e-9, (k, l, rms, rms_cv)
        np.testing.assert_allclose(sm[:, :3] @ sm[:, :3].T, np.eye(3), atol=1e-12)
        if l < L:
            dR = np.abs(sm[:, :3] - p_ref[:, :3]).max()
            dt = np.abs(sm[:, 3] - p_ref[:, 3]).max() / np.linalg.norm(p_ref[:, 3])
            assert dR < 1e-7 and dt < 1e-7, (k, l, dR, dt)
            worst.update(corners_ulp=max(worst['corners_ulp'], ulps(c, c_ref)), dR=max(worst['dR'], dR), dt=max(worst['dt'], dt),
                         rms_px=max(worst['rms_px'], rms_cv))
        cases += 1
    print(f'num {num} std {std}: {cases} cases, worst vs OpenCV', worst)
    assert cases >= 100 and worst['rms_px'] > 0.5          # the averaging noise reaches the 0 - 2 px range
    # the special lanes do exercise the clamp / a negative depth
    clamp, behind = tracks[L][0], tracks[L + 1][0]
    assert np.abs((BBOX @ clamp[:, :3].T + clamp[:, 3])[:, 2]).min() < 1e-4
    assert (BBOX @ behind[:, :3].T + behind[:, 3])[:, 2].min() < 0


@pytest.fixture(scope='module')
def golden():
    return np.load(os.path.join(HERE, 'golden', 'track_golden.npz'))


def test_oracle_reproduces_reference_tracking_golden(golden):
    """oracle/track.py on the reference's own poses reproduces the reference's corners, averages and PnP poses."""
    G = golden
    out = T.smooth_sequence(G['track.bbox'], G['track.pose'], G['track.K'], int(G['track.num']), float(G['track.std']))
    for k, (c, w, p) in enumerate(out):
        np.testing.assert_array_equal(c, G['track.corners'][k])
        np.testing.assert_array_equal(w, G['track.wpts'][k])
        np.testing.assert_allclose(p, G['track.pnp'][k], rtol=0, atol=1e-12)


def test_host_twin_reproduces_reference_tracking_golden(golden):
    """The kernel's code fed the reference's per-frame poses gives the reference's corners (float32, <= 2 ulps), weighted
    points and smoothed poses (R within 1e-7, t within 1e-7 relative, reprojection no worse than OpenCV's)."""
    G = golden
    num, std, K, bbox = int(G['track.num']), float(G['track.std']), G['track.K'], G['track.bbox']
    assert G['track.pose'].dtype == np.float32 and bbox.shape == (8, 3) and len(G['track.pose']) == 8
    w, ws = glue.smoothing_weights(num, std)
    hist, cnt = np.zeros((1, num, 8, 2), np.float32), np.zeros(1, np.int32)
    for k, pose in enumerate(G['track.pose']):
        c, wp, sm = glue.host_track_smooth(glue.check_bbox(bbox), pose[None].astype(np.float64), glue.cameras(K[None]), w, ws, hist, cnt)
        assert ulps(c[0], G['track.corners'][k]) <= 2, k
        np.testing.assert_allclose(wp[0], G['track.wpts'][k], rtol=1e-7, atol=0)
        p_ref = G['track.pnp'][k]
        assert np.abs(sm[0, :, :3] - p_ref[:, :3]).max() < 1e-7, k
        assert np.abs(sm[0, :, 3] - p_ref[:, 3]).max() / np.linalg.norm(p_ref[:, 3]) < 1e-7, k
        wk = G['track.wpts'][k]
        assert T.reprojection_rms(bbox, wk, sm[0], K) <= T.reprojection_rms(bbox, wk, p_ref, K) + 1e-9


def test_bbox_checks():
    """A box the smoothing PnP cannot take is refused before anything runs."""
    from gen6d_b200.tracker import Gen6DTracker
    flat = BBOX.copy()
    flat[:, 2] = 0.3                                   # all corners in one plane
    thin = BBOX.copy()
    thin[:, 2] *= 1e-3                                 # nearly planar: below OpenCV's 1e-3 singular-value ratio
    for bad in (flat, thin, BBOX[:7], np.zeros((8, 3)), np.full((8, 3), np.nan), BBOX.reshape(4, 6)):
        with pytest.raises(ValueError):
            glue.check_bbox(bad)
        with pytest.raises(ValueError):
            Gen6DTracker(None, bbox_3d=bad)
    assert glue.check_bbox(BBOX.astype(np.float64)).dtype == np.float32
    with pytest.raises(ValueError):
        Gen6DTracker(None, bbox_3d=BBOX, smooth_num=0)


def test_smoothing_weights_match_predict_py():
    for num, std in ((5, 2.5), (10, 10.0), (1, 1.0)):
        w, ws = glue.smoothing_weights(num, std)
        assert w[-1] == 1.0 and len(w) == len(ws) == num
        ref = np.exp(-(np.arange(num) / std) ** 2)[::-1]
        np.testing.assert_array_equal(w, ref)
        for n in range(1, num + 1):
            assert ws[n - 1] == np.sum(ref[-n:])
