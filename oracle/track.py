"""numpy / OpenCV restatement of the pose smoothing of the reference's video tracker (predict.py), the oracle of
csrc/track.cu (g6d_track_smooth):
  * project_points   -- utils/base_utils.py:256-265
  * weighted_pts     -- predict.py:18-26
  * pnp              -- utils/pose_utils.py:246-279 (cv2.solvePnP, SOLVEPNP_ITERATIVE, zero distortion)
  * bbox_corners     -- utils/draw_utils.py:258-270 pts_range_to_bbox_pts
  * smooth_sequence  -- predict.py:63-71: one smoothed pose per frame of a pose sequence
"""
import cv2
import numpy as np


def project_points(pts, RT, K):
    pts = np.matmul(pts, RT[:, :3].transpose()) + RT[:, 3:].transpose()
    pts = np.matmul(pts, K.transpose())
    dpt = pts[:, 2]
    mask0 = (np.abs(dpt) < 1e-4) & (np.abs(dpt) > 0)
    if np.sum(mask0) > 0:
        dpt[mask0] = 1e-4
    mask1 = (np.abs(dpt) > -1e-4) & (np.abs(dpt) < 0)
    if np.sum(mask1) > 0:
        dpt[mask1] = -1e-4
    return pts[:, :2] / dpt[:, None], dpt


def weighted_pts(pts_list, weight_num=10, std_inv=10):
    weights = np.exp(-(np.arange(weight_num) / std_inv) ** 2)[::-1]
    pose_num = len(pts_list)
    if pose_num < weight_num:
        weights = weights[-pose_num:]
    else:
        pts_list = pts_list[-weight_num:]
    return np.sum(np.asarray(pts_list) * weights[:, None, None], 0) / np.sum(weights)


def pnp(points_3d, points_2d, camera_matrix):
    dist_coeffs = np.zeros(shape=[8, 1], dtype='float64')
    points_2d = np.ascontiguousarray(points_2d.astype(np.float64))
    points_3d = np.ascontiguousarray(points_3d.astype(np.float64))
    _, R_exp, t = cv2.solvePnP(points_3d, points_2d, camera_matrix.astype(np.float64), dist_coeffs, flags=cv2.SOLVEPNP_ITERATIVE)
    R, _ = cv2.Rodrigues(R_exp)
    return np.concatenate([R, t], axis=-1)


def bbox_corners(max_pt, min_pt):
    maxx, maxy, maxz = max_pt
    minx, miny, minz = min_pt
    return np.asarray([[minx, miny, minz], [minx, maxy, minz], [maxx, maxy, minz], [maxx, miny, minz],
                       [minx, miny, maxz], [minx, maxy, maxz], [maxx, maxy, maxz], [maxx, miny, maxz]])


def reprojection_rms(points_3d, points_2d, pose, K):
    """RMS pixel distance of the float64 projections of points_3d under pose to points_2d."""
    X = np.asarray(points_3d, np.float64) @ pose[:, :3].T + pose[:, 3]
    p = X @ np.asarray(K, np.float64).T
    return float(np.sqrt(np.mean(np.sum((p[:, :2] / p[:, 2:] - points_2d) ** 2, 1))))


def smooth_sequence(bbox, poses, K, num=5, std=2.5):
    """predict.py:63-71 over a sequence of poses: per frame (projected corners, weighted points, pnp pose)."""
    hist, out = [], []
    for pose in poses:
        pts, _ = project_points(bbox, pose, K)
        hist.append(pts)
        w = weighted_pts(hist, weight_num=num, std_inv=std)
        out.append((pts, w, pnp(bbox, w, K)))
    return out
