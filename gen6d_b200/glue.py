"""Tables and call wrappers of the device-side camera algebra (csrc/glue.cu, include/gen6d_b200.h g6d_glue_*).

Between the stages of a prediction the reference's estimator does small camera computations on the host
(estimator.py:176-214).  geometry.py restates them in numpy; csrc/glue_math.cuh restates them once more as
__host__ __device__ code so that a batched prediction can stay on the GPU from the uploaded frames to the final
poses.  This module builds what those kernels read:
  * cameras(que_Ks): per-frame constants that depend on K only (K, np.linalg.inv(K), (K00 + K11) / 2, each evaluated
    by numpy in K's own dtype, handed over as float64 values);
  * selector_refs(ref_info): per selector reference view, what poses_from_similarity needs of it;
  * refiner_views(database, ref_ids, ...): the pose-independent view table of geometry.NormalizedView, the FPS
    re-spread subset with its viewing directions, and the unit-sphere normalisation.
The `host_*` functions run the library's *_host entry points on numpy arrays: same code as the kernels, no GPU --
tests/test_glue.py pins them against geometry.py.
"""
import ctypes as C

import numpy as np

from . import _lib
from . import geometry as G

JOB = G.WARP_JOB


def cameras(que_Ks):
    """[qn,3,3] intrinsics (any float dtype) -> float64 [qn,20] = g6d_glue_camera records."""
    Ks = np.asarray(que_Ks)
    out = np.zeros((len(Ks), 20), np.float64)
    out[:, :9] = Ks.reshape(len(Ks), 9)
    out[:, 9:18] = np.linalg.inv(Ks).reshape(len(Ks), 9)
    f = (Ks[:, 0, 0] + Ks[:, 1, 1]) / 2
    out[:, 18], out[:, 19] = f, f ** 2
    return out


def selector_refs(ref_info):
    """estimator.ref_info -> arrays of g6d_glue_refs (what geometry.poses_from_similarity reads per reference view)."""
    poses, Ks = np.asarray(ref_info['poses']), np.asarray(ref_info['Ks'])
    center = np.asarray(ref_info['center'], np.float64)
    return {'poses': np.ascontiguousarray(poses.reshape(len(poses), 12), np.float64),
            'cen': np.ascontiguousarray(G._project_center_batch(center, poses, Ks), np.float64),
            'f': np.ascontiguousarray((Ks[:, 0, 0] + Ks[:, 1, 1]) / 2, np.float64),
            'dist': np.asarray([np.linalg.norm(G.camera_center(p) - center) for p in poses], np.float64),
            'center': center}


def refiner_views(database, ref_ids, size=128, ref_num=6, margin=0.05):
    """The refiner's view tables (g6d_glue_views minus the image addresses) for refine_problems(ref_even=True)."""
    view = G._normalized_view(database)
    ids = list(ref_ids)
    tab = view.view_table(ids, size, margin, prefill=ids)
    center = view.object_center()
    ids_e, _, dirs = view.even_subset(ids, min(128, len(ids)), center)
    row = {i: k for k, i in enumerate(ids)}
    n = len(ids)
    return {'ids': ids, 'view': view,
            'poses': np.ascontiguousarray(tab['poses'].reshape(n, 12), np.float64),
            'R_look': np.ascontiguousarray(tab['R_look'].reshape(n, 9), np.float64),
            'RlookR': np.ascontiguousarray(tab['RlookR'].reshape(n, 9), np.float64),
            'f': np.ascontiguousarray(tab['f'], np.float64),
            'Kinv': np.ascontiguousarray(tab['Kinv'].reshape(n, 9), np.float64),
            'even_idx': np.asarray([row[i] for i in ids_e], np.int32),
            'even_dirs': np.ascontiguousarray(dirs, np.float32),
            'norm_scale': float(view.scale), 'norm_offset': np.asarray(view.offset, np.float32),
            'size_scale': np.float32(size * (1 - margin) / view.object_diameter()), 'size': size, 'ref_num': ref_num}


# ------------------------------------------------------------------------------------------ struct packing
def _ptr(a):
    return a.ctypes.data if isinstance(a, np.ndarray) else int(a)


def refs_struct(arr):
    """arr: dict of numpy arrays (host entry points) or of device addresses."""
    s = _lib.GlueRefs()
    s.poses, s.cen, s.f, s.dist = _ptr(arr['poses']), _ptr(arr['cen']), _ptr(arr['f']), _ptr(arr['dist'])
    s.center[:] = [float(v) for v in arr['center']]
    return s


def views_struct(arr, tables, src=0, rows=0, cols=0):
    """arr: addresses (numpy arrays or device pointers) of the per-view arrays; tables: the refiner_views() dict."""
    s = _lib.GlueViews()
    for k in ('poses', 'R_look', 'RlookR', 'f', 'Kinv', 'even_idx', 'even_dirs'):
        setattr(s, k, _ptr(arr[k]))
    s.src, s.rows, s.cols = _ptr(src), _ptr(rows), _ptr(cols)
    s.n_views, s.n_even, s.ref_num, s.size = len(tables['ids']), len(tables['even_idx']), tables['ref_num'], tables['size']
    s.norm_scale = tables['norm_scale']
    s.norm_offset[:] = [float(v) for v in tables['norm_offset']]
    s.size_scale = float(tables['size_scale'])
    return s


# ------------------------------------------------------------------------------------------ host entry points (tests)
def host_detection_jobs(det_out, rows, cols, size, frame_ptr=0):
    det = np.ascontiguousarray(det_out, np.float32)
    jobs = np.zeros(len(det), JOB)
    _lib.check(_lib.lib().g6d_glue_detection_jobs_host(det.ctypes.data, frame_ptr, rows, cols, len(det), size, jobs.ctypes.data),
               'g6d_glue_detection_jobs_host')
    return jobs


def host_initial_poses(det_out, sel_idx, sel_out, refs, cams):
    det, idx = np.ascontiguousarray(det_out, np.float32), np.ascontiguousarray(sel_idx, np.int64)
    so, cams = np.ascontiguousarray(sel_out, np.float32), np.ascontiguousarray(cams, np.float64)
    poses = np.zeros((len(det), 3, 4), np.float64)
    st = refs_struct(refs)
    _lib.check(_lib.lib().g6d_glue_initial_poses_host(det.ctypes.data, idx.ctypes.data, so.ctypes.data, C.byref(st), cams.ctypes.data,
                                                      len(det), poses.ctypes.data), 'g6d_glue_initial_poses_host')
    return poses


def host_refine_problems(tables, cams, poses, poses_are_f32, rows, cols, frame_ptr=0, src=None, img_rows=None, img_cols=None):
    n, R = len(poses), tables['ref_num']
    nv = len(tables['ids'])
    src = np.zeros(nv, np.uint64) if src is None else np.ascontiguousarray(src, np.uint64)
    img_rows = np.zeros(nv, np.int32) if img_rows is None else np.ascontiguousarray(img_rows, np.int32)
    img_cols = np.zeros(nv, np.int32) if img_cols is None else np.ascontiguousarray(img_cols, np.int32)
    st = views_struct(tables, tables, src, img_rows, img_cols)
    cams, poses = np.ascontiguousarray(cams, np.float64), np.ascontiguousarray(poses, np.float64)
    out = {'jobs': np.zeros(n * (R + 1), JOB), 'que_K': np.zeros((n, 3, 3), np.float32), 'que_pose': np.zeros((n, 3, 4), np.float32),
           'pose_rect': np.zeros((n, 3, 4), np.float32), 'ref_Ks': np.zeros((n, R, 3, 3), np.float32),
           'ref_poses': np.zeros((n, R, 3, 4), np.float32), 'ref_rows': np.zeros((n, R), np.int32)}
    _lib.check(_lib.lib().g6d_glue_refine_problems_host(C.byref(st), cams.ctypes.data, frame_ptr, rows, cols, poses.ctypes.data,
                                                        int(poses_are_f32), n, *[out[k].ctypes.data for k in
                                                                                 ('jobs', 'que_K', 'que_pose', 'pose_rect', 'ref_Ks',
                                                                                  'ref_poses', 'ref_rows')]),
               'g6d_glue_refine_problems_host')
    return out


def host_apply_refinements(tables, prob, net_out):
    st = views_struct(tables, tables)
    net = np.ascontiguousarray(net_out, np.float32)
    poses = np.zeros((len(net), 3, 4), np.float64)
    _lib.check(_lib.lib().g6d_glue_apply_refinements_host(C.byref(st), prob['que_pose'].ctypes.data, prob['que_K'].ctypes.data,
                                                          prob['pose_rect'].ctypes.data, net.ctypes.data, len(net), poses.ctypes.data),
               'g6d_glue_apply_refinements_host')
    return poses


# ------------------------------------------------------------------------------------------ pose smoothing (csrc/track.cu)
def smoothing_weights(num, std):
    """predict.py:19-23: weights = exp(-(arange(num) / std) ** 2)[::-1] (newest last, weight 1) and wsum[n - 1] = the sum
    of the last n of them, the normaliser of a history of n < num projections -- both evaluated by numpy, so that the
    kernel's average divides by exactly what the reference divides by."""
    w = np.ascontiguousarray(np.exp(-(np.arange(num) / std) ** 2)[::-1], np.float64)
    return w, np.asarray([np.sum(w[-n:]) for n in range(1, num + 1)], np.float64)


def check_bbox(bbox_3d):
    """bbox_3d -> float32 [8,3]; ValueError unless it is 8 x 3 and non-coplanar by cv::solvePnP's test (the smallest over
    the middle singular value of the centred points' 3x3 scatter matrix >= 1e-3; below it OpenCV takes its planar
    homography branch, which the smoothing kernel does not implement)."""
    b = np.asarray(bbox_3d)
    if b.shape != (8, 3) or not np.all(np.isfinite(b)):
        raise ValueError(f'bbox_3d must be 8 x 3 finite corners, got shape {b.shape}')
    b = np.ascontiguousarray(b, np.float32)
    c = b.astype(np.float64) - b.astype(np.float64).mean(0)
    w = np.linalg.svd(c.T @ c, compute_uv=False)
    if not w[1] > 0 or w[2] / w[1] < 1e-3:
        raise ValueError('bbox_3d is degenerate or planar: the smoothing PnP needs non-coplanar corners')
    return b


def host_track_smooth(bbox, poses, cams, weights, wsum, hist, count):
    """g6d_track_smooth_host: the kernel's code on numpy arrays.  hist f32 [M,num,8,2] and count i32 [M] are updated in
    place.  Returns (corners f32 [M,8,2], averaged corners f64 [M,8,2], smoothed poses f64 [M,3,4])."""
    bbox = np.ascontiguousarray(bbox, np.float32)
    poses = np.ascontiguousarray(np.asarray(poses, np.float64).reshape(-1, 12))
    cams = np.ascontiguousarray(cams, np.float64)
    weights, wsum = np.ascontiguousarray(weights, np.float64), np.ascontiguousarray(wsum, np.float64)
    assert hist.dtype == np.float32 and hist.flags.c_contiguous and count.dtype == np.int32 and count.flags.c_contiguous
    M = len(poses)
    corners, wpts, smoothed = np.zeros((M, 8, 2), np.float32), np.zeros((M, 8, 2), np.float64), np.zeros((M, 3, 4), np.float64)
    _lib.check(_lib.lib().g6d_track_smooth_host(bbox.ctypes.data, poses.ctypes.data, cams.ctypes.data, weights.ctypes.data,
                                                wsum.ctypes.data, M, len(weights), hist.ctypes.data, count.ctypes.data,
                                                corners.ctypes.data, wpts.ctypes.data, smoothed.ctypes.data), 'g6d_track_smooth_host')
    return corners, wpts, smoothed
