"""The synthetic video of the tracking goldens (make_golden_track.py) and tests: a smooth camera path that starts at the
pose of query view '11' of the synthetic database, with predict.py's pseudo intrinsics f = sqrt(h^2 + w^2)."""
import numpy as np

N_FRAMES = 8


def _rot_z(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0.], [s, c, 0.], [0., 0., 1.]])


def track_path(db, n=N_FRAMES, start='11'):
    """-> (poses float32 [n,3,4], K float32 [3,3]): the object turns 0.03 rad per frame about the database's up axis
    (through the object centre at the origin) while the camera backs off by 1 % per frame."""
    p0 = db.get_pose(start).astype(np.float64)
    poses = [np.concatenate([p0[:, :3] @ _rot_z(0.03 * k), p0[:, 3:] * (1 + 0.01 * k)], 1).astype(np.float32) for k in range(n)]
    h, w = db.h, db.w
    f = np.sqrt(h ** 2 + w ** 2)
    return poses, np.asarray([[f, 0, w / 2], [0, f, h / 2], [0, 0, 1]], np.float32)
