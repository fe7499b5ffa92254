"""Gen6DTracker on the B200: the smoothing kernel against its host twin, start() against predict_batch / predict(pose_init),
teacher-forced steps against the refiner's batched refinement and against the reference's tracking video, carried poses,
and the captured-graph housekeeping."""
import os

import numpy as np
import pytest

from golden import cases
from golden.track_path import track_path

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
E = np.load(os.path.join(HERE, 'golden', 'est_golden.npz'))
TG = np.load(os.path.join(HERE, 'golden', 'track_golden.npz'))
S = np.load(os.path.join(HERE, 'golden', 'sens_golden.npz'))


@pytest.fixture(scope='module')
def est():
    from gen6d_b200.synthetic import build_estimator
    return build_estimator()


def videos(db, M, n=4):
    """M lanes of the synthetic tracking video, each starting at its own database view -> (frames [n][M], Ks, paths [n,M])."""
    paths, K = zip(*[track_path(db, n=n, start=str(11 + 2 * j)) for j in range(M)])
    frames = [np.stack([db.render(paths[j][k], K[j]) for j in range(M)]) for k in range(n)]
    return frames, np.stack(K), np.stack([np.stack(p) for p in paths], 1)


def perturb(poses, seed, rot=0.02, trans=0.03):
    import cv2
    rng = np.random.RandomState(seed)
    out = []
    for p in poses.reshape(-1, 3, 4):
        R = cv2.Rodrigues(rng.randn(3) * rot)[0] @ p[:, :3]
        out.append(np.concatenate([R, p[:, 3:] * (1 + trans * rng.randn())], 1))
    return np.stack(out).reshape(poses.shape).astype(np.float32)


def bbox_of(db):
    from oracle import track as T
    pts = db.object_point_cloud
    return T.bbox_corners(pts.max(0), pts.min(0)).astype(np.float32)


def test_kernel_equals_host_twin():
    """g6d_track_smooth on the device = g6d_track_smooth_host bit for bit, ring wrap and several lanes included."""
    import torch
    from gen6d_b200 import glue, ops
    from test_track_cpu import BBOX, noisy_track, special_track
    for num, std in ((5, 2.5), (10, 10.0)):
        rng = np.random.RandomState(num)
        L = 12
        Ks = [np.array([[f, 0, 320], [0, f, 240], [0, 0, 1]], np.float32) for f in 500 + 400 * rng.rand(L)]
        tracks = [noisy_track(rng, num + 3, float(Ks[l][0, 0]), 25.0) for l in range(L)]
        tracks += [special_track(num + 3, 'clamp'), special_track(num + 3, 'behind')]
        Ks += [Ks[0], Ks[0]]
        M = len(tracks)
        w, ws = glue.smoothing_weights(num, std)
        cams = glue.cameras(np.stack(Ks))
        hist, cnt = np.zeros((M, num, 8, 2), np.float32), np.zeros(M, np.int32)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        d_hist, d_cnt, d_args = dev(hist), dev(cnt), [dev(BBOX), None, dev(cams), dev(w), dev(ws)]
        for k in range(num + 3):
            poses = np.stack([t[k] for t in tracks]).astype(np.float64).reshape(M, 12)
            c, wp, sm = glue.host_track_smooth(BBOX, poses, cams, w, ws, hist, cnt)
            d_args[1] = dev(poses)
            dc, dw, ds = [t.cpu().numpy() for t in ops.track_smooth(*d_args, d_hist, d_cnt)]
            np.testing.assert_array_equal(dc, c)
            np.testing.assert_array_equal(dw, wp)
            np.testing.assert_array_equal(ds.reshape(M, 3, 4), sm)
            np.testing.assert_array_equal(d_hist.cpu().numpy(), hist)
            np.testing.assert_array_equal(d_cnt.cpu().numpy(), cnt)


def test_start_matches_predict_batch(est):
    """start() without poses is predict_batch's device-resident prediction: same detections, selections and pose chain."""
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    ids = db.get_img_ids()[:4]
    imgs, Ks = np.stack([db.get_image(i) for i in ids]), np.stack([db.get_K(i) for i in ids])
    assert e.cfg['device_glue']
    want_poses, want = e.predict_batch(list(imgs), list(Ks))
    poses, smoothed, inter = Gen6DTracker(e, bbox_of(db)).start(imgs, Ks)
    for k in ('det_position', 'det_scale_r2q', 'sel_ref_idx', 'sel_angle_r2q', 'det_que_img', 'sel_scores'):
        np.testing.assert_array_equal(inter[k], want[k], err_msg=k)
    for a, b in zip(inter['refine_poses'], want['refine_poses']):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(poses, want_poses)
    assert smoothed.shape == (4, 3, 4) and smoothed.dtype == np.float64


def test_start_from_pose_matches_reference_tracking(est):
    """start(frame, K, poses=...) = predict(pose_init=...): cfg['refine_iter'] refinements, within
    test_tracking_refinement_matches_reference's bounds of the reference's chain."""
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    q = str(int(E['est.query_id']))
    tr = Gen6DTracker(e)
    pose, smoothed, inter = tr.start(db.get_image(q)[None], db.get_K(q)[None], poses=E['est.track_init'][None])
    assert smoothed is None
    got, want = np.stack([p[0] for p in inter['refine_poses']], 0), E['est.track_poses']
    err_r = np.abs(got[:, :, :3] - want[:, :, :3]).reshape(len(got), -1).max(1)
    err_t = np.abs(got[:, :, 3] - want[:, :, 3]).max(1) / np.linalg.norm(want[:, :, 3], axis=1)
    print('start(poses) vs reference tracking chain: per-iteration max |dR|', err_r, 'relative |dt|', err_t)
    np.testing.assert_allclose(got[:, :, :3], want[:, :, :3], atol=1e-2)
    assert (err_t < 1e-2).all()
    np.testing.assert_array_equal(pose[0], got[-1])
    host, _ = e.predict(db.get_image(q), db.get_K(q), pose_init=E['est.track_init'])
    print('start(poses) vs predict(pose_init), max |dpose|', float(np.abs(pose[0] - host).max()))


@pytest.mark.parametrize('M', [1, 4])
def test_teacher_forced_steps_equal_refine_batch(est, M):
    """step(frames, poses=P) = refiner.refine_batch(frames, Ks, P) (one refinement), to the device-vs-host bound."""
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    frames, Ks, paths = videos(db, M)
    tr = Gen6DTracker(e, bbox_of(db))
    tr.start(frames[0], Ks, poses=perturb(paths[0], 1))
    for k in range(1, len(frames)):
        P = perturb(paths[k], 10 + k)
        got, _ = tr.step(frames[k], poses=P)
        want = e.refiner.refine_batch(e.detector.upload_frame(list(frames[k])), list(Ks), P, size=128, ref_num=6, ref_even=True)
        d = float(np.abs(got - want).max())
        print(f'M={M} step {k}: teacher-forced step vs refine_batch, max |dpose|', d)
        assert d < 2e-4


def test_steps_carry_the_pose(est):
    """An un-forced step starts from the previous step's output: re-seeding a second tracker with those outputs gives the
    same poses bit for bit."""
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    frames, Ks, paths = videos(db, 2, n=5)
    a, b = Gen6DTracker(e, bbox_of(db)), Gen6DTracker(e, bbox_of(db))
    init = perturb(paths[0], 3)
    prev, _, _ = a.start(frames[0], Ks, poses=init)
    b.start(frames[0], Ks, poses=init)
    for k in range(1, len(frames)):
        out, _ = a.step(frames[k])
        forced, _ = b.step(frames[k], poses=prev)
        np.testing.assert_array_equal(out, forced)
        assert not np.array_equal(out, prev)
        prev = out


def test_teacher_forced_reference_video(est):
    """Frames 1-7 of the reference's tracking video, each step forced with the reference's input pose, give the
    reference's refined poses within the est.track bounds (1e-2 on R, 1e-2 relative on t)."""
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    path, K = track_path(db)
    np.testing.assert_array_equal(np.stack(path), TG['track.path'])
    np.testing.assert_array_equal(K, TG['track.K'])
    frames = [db.render(p, K)[None] for p in path]
    tr = Gen6DTracker(e, TG['track.bbox'], smooth_num=int(TG['track.num']), smooth_std=float(TG['track.std']))
    tr.start(frames[0], K[None], poses=TG['track.pose'][:1])
    err_r, err_t = [], []
    for k in range(1, len(frames)):
        got, _ = tr.step(frames[k], poses=TG['track.in_pose'][k][None])
        want = TG['track.pose'][k]
        err_r.append(float(np.abs(got[0, :, :3] - want[:, :3]).max()))
        err_t.append(float(np.abs(got[0, :, 3] - want[:, 3]).max() / np.linalg.norm(want[:, 3])))
    print('reference video frames 1-7, teacher-forced: max |dR|', np.round(err_r, 6), 'relative |dt|', np.round(err_t, 6))
    assert max(err_r) < 1e-2 and max(err_t) < 1e-2


def test_smoothing_on_device_equals_host_twin_of_run(est):
    """The smoothed poses of a tracked run (full start, then un-forced steps) = the host twin applied to the run's poses."""
    from gen6d_b200 import glue
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    frames, Ks, _ = videos(db, 3, n=8)
    bbox = bbox_of(db)
    tr = Gen6DTracker(e, bbox, smooth_num=5, smooth_std=2.5)
    runs = [tr.start(frames[0], Ks)[:2]] + [tr.step(f) for f in frames[1:]]
    w, ws = glue.smoothing_weights(5, 2.5)
    hist, cnt = np.zeros((3, 5, 8, 2), np.float32), np.zeros(3, np.int32)
    for poses, smoothed in runs:
        _, _, want = glue.host_track_smooth(bbox, poses.astype(np.float64), glue.cameras(Ks), w, ws, hist, cnt)
        np.testing.assert_array_equal(smoothed, want)
    assert cnt.tolist() == [8, 8, 8]


def test_graph_housekeeping(est):
    """Replays are deterministic, two trackers on one estimator stepped alternately give their solo results, bad calls
    raise before anything runs, and build() on another database forces a re-capture."""
    from gen6d_b200.synthetic import synthetic_database
    from gen6d_b200.tracker import Gen6DTracker
    e, db = est
    fa, Ka, pa = videos(db, 2, n=4)
    fb, Kb, pb = videos(db, 3, n=4)
    bbox = bbox_of(db)

    def solo(frames, Ks, paths):
        tr = Gen6DTracker(e, bbox)
        out = [tr.start(frames[0], Ks, poses=paths[0])[:2]]
        return out + [tr.step(f) for f in frames[1:]]
    sa, sb = solo(fa, Ka, pa), solo(fb, Kb, pb)
    for x, y in zip(sa, solo(fa, Ka, pa)):                      # deterministic replays
        np.testing.assert_array_equal(x[0], y[0])
        np.testing.assert_array_equal(x[1], y[1])
    ta, tb = Gen6DTracker(e, bbox), Gen6DTracker(e, bbox)
    alt_a, alt_b = [ta.start(fa[0], Ka, poses=pa[0])[:2]], [tb.start(fb[0], Kb, poses=pb[0])[:2]]
    for k in range(1, 4):
        alt_a.append(ta.step(fa[k]))
        alt_b.append(tb.step(fb[k]))
    for solo_r, alt_r in ((sa, alt_a), (sb, alt_b)):
        for x, y in zip(solo_r, alt_r):
            np.testing.assert_array_equal(x[0], y[0])
            np.testing.assert_array_equal(x[1], y[1])
    with pytest.raises(RuntimeError):
        Gen6DTracker(e, bbox).step(fa[1])
    with pytest.raises(ValueError):
        ta.step(fb[1])                                          # 3 lanes after a 2-lane start
    with pytest.raises(ValueError):
        ta.step(fa[1][:, :240])                                 # another frame size
    # a rebuild on another object bumps the estimator's generation: the tracker's graphs are captured anew
    step_stage = [s for k, s in ta.stages.stages.items() if k[0] == 'step']
    assert len(step_stage) == 1
    try:
        e.build(synthetic_database(seed=8), 'all')
        ta.step(fa[1])
        again = [s for k, s in ta.stages.stages.items() if k[0] == 'step']
        assert len(again) == 1 and again[0] is not step_stage[0]
    finally:
        e.build(db, 'all')
    out, _ = ta.step(fa[1])
    assert np.isfinite(out).all()
