"""Gen6DTracker: the reference's video tracking loop (predict.py:47-72) with the pose kept on the device.

The reference tracks an object through a video with one estimator: the first frame runs the full prediction (detect ->
select -> refine_iter refinements), every later frame only refines the previous frame's pose once, and the output is
smoothed by projecting the object's 3-D box with each pose, averaging the last `num` projections with weights
exp(-(k / std) ** 2) and solving PnP for the average (predict.py:18-26, 63-71).

Here M independent videos run in lockstep, one lane each.  A tracked step is one captured CUDA graph per lane count:
refine_iter x (g6d_glue_refine_problems -> refiner -> g6d_glue_apply_refinements) from the carried poses, then the
smoothing kernel (csrc/track.cu) on the per-lane history ring.  The carried poses, the intrinsics and the history stay on
the device; a step moves the frames in and the [M,12] poses (+ smoothed poses) out, nothing else.

    tr = Gen6DTracker(estimator, bbox_3d, smooth_num=5, smooth_std=2.5, refine_iter=1)
    poses, smoothed, inter = tr.start(frames_u8[M,h,w,3], Ks[M,3,3])     # first frames: full prediction
    poses, smoothed = tr.step(next_frames_u8[M,h,w,3])                   # every later frame
"""
import numpy as np
import torch

from . import glue
from . import ops
from .graphs import StageCache


class Gen6DTracker:
    def __init__(self, estimator, bbox_3d=None, smooth_num=5, smooth_std=2.5, refine_iter=1):
        """estimator: a built Gen6DEstimator (its networks, reference state and cfg['refine_iter'] for the first frame).
        bbox_3d: [8,3] object box corners (utils/draw_utils.py pts_range_to_bbox_pts order) or None for no smoothing.
        smooth_num / smooth_std: predict.py's --num / --std.  refine_iter: refinements per tracked frame."""
        self.est = estimator
        self.bbox = None if bbox_3d is None else glue.check_bbox(bbox_3d)
        if int(smooth_num) < 1 or not float(smooth_std) > 0:
            raise ValueError('smooth_num must be >= 1 and smooth_std > 0')
        self.num, self.std, self.refine_iter = int(smooth_num), float(smooth_std), int(refine_iter)
        self.weights, self.wsum = glue.smoothing_weights(self.num, self.std)
        self.stages = StageCache()
        self._state = {}             # lane count -> device state the captured graphs read and write
        self._gen = None
        self._shape = None           # frames shape [M,h,w,3] of the current videos

    # ------------------------------------------------------------------ device state and graphs
    def _lanes(self, M):
        S = self._state.get(M)
        if S is None:
            dev = self.est.detector.device
            S = {'poses': torch.zeros(M, 12, device=dev, dtype=torch.float64),
                 'cams': torch.zeros(M, 20, device=dev, dtype=torch.float64),
                 'hist': torch.zeros(M, self.num, 8, 2, device=dev, dtype=torch.float32),
                 'count': torch.zeros(M, device=dev, dtype=torch.int32)}
            if self.bbox is not None:
                S['bbox'] = torch.from_numpy(self.bbox).to(dev)
                S['weights'], S['wsum'] = torch.from_numpy(self.weights).to(dev), torch.from_numpy(self.wsum).to(dev)
            self._state[M] = S
        return S

    def _glue(self):
        """The estimator's device tables; graphs captured against an older generation of them are dropped."""
        est = self.est
        if not est._glue_possible():
            raise RuntimeError('Gen6DTracker needs the device-resident path: a refiner, a capturable selector and '
                               "cfg['host_warps'] = False")
        st = est._glue_state()
        gen = est._generation()
        if gen != self._gen:
            self.stages.clear()
            self._gen = gen
        return st

    def _refine(self, st, S, frames, poses, iters, first_f32):
        """iters x (problems -> refiner -> update) from poses [M,12] float64 on the device."""
        refine, R = self.est.refiner._refine_warped(128), st['tables']['ref_num']
        for it in range(iters):
            jobs, que_K, que_pose, rect, ref_Ks, ref_poses, _ = ops.glue_refine_problems(st['views'], R, S['cams'], frames, poses,
                                                                                         first_f32 or it > 0)
            out = refine(jobs, que_K, que_pose, ref_Ks, ref_poses)
            poses = ops.glue_apply_refinements(st['views'], que_pose, que_K, rect, out)
        return poses

    def _finish(self, S, poses, reset):
        """Carry `poses`, run the smoothing kernel -> [M,12] or [M,24] (poses | smoothed) for one D2H read."""
        if poses is not S['poses']:
            S['poses'].copy_(poses)
        if reset:
            S['count'].zero_()
        if self.bbox is None:
            return S['poses'].clone()
        _, _, smoothed = ops.track_smooth(S['bbox'], S['poses'], S['cams'], S['weights'], S['wsum'], S['hist'], S['count'])
        return torch.cat([S['poses'], smoothed], 1)

    def _state_list(self, S):
        return [S['poses'], S['hist'], S['count']]

    def _split(self, out, M):
        out = self.est.detector._to_host(out)
        poses = out[:, :12].reshape(M, 3, 4).astype(np.float32)
        return poses, (out[:, 12:].reshape(M, 3, 4) if self.bbox is not None else None)

    def _upload(self, frames):
        frames = [np.asarray(f) for f in frames]
        if not frames or any(f.dtype != np.uint8 or f.ndim != 3 or f.shape[2] != 3 or f.shape != frames[0].shape for f in frames):
            raise ValueError('frames must be M >= 1 uint8 [h,w,3] images of one size')
        return (len(frames),) + frames[0].shape, frames

    # ------------------------------------------------------------------ public API
    def start(self, frames, Ks, poses=None):
        """First frames of M videos.  frames: uint8 [M,h,w,3] (or a list); Ks: [M,3,3], fixed per lane from here on.
        poses None: the full device-resident prediction of predict_batch (detect -> select -> cfg['refine_iter']
        refinements); otherwise cfg['refine_iter'] refinements from the given [M,3,4] poses (predict(pose_init=...);
        float32 poses are refined as float32, as the reference does with a refined pose).  The smoothing history is
        reset.  Returns (poses float32 [M,3,4], smoothed float64 [M,3,4] or None, inter) with inter = predict_batch's
        inter dict (poses None) or {'refine_poses': [...]}."""
        shape, frames = self._upload(frames)
        M = shape[0]
        Ks = np.asarray(Ks)
        if Ks.shape != (M, 3, 3):
            raise ValueError(f'Ks must be [{M},3,3], got {Ks.shape}')
        if poses is not None:
            poses = np.asarray(poses)
            if poses.shape != (M, 3, 4) or poses.dtype not in (np.float32, np.float64):
                raise ValueError(f'poses must be float32 / float64 [{M},3,4]')
        st = self._glue()
        est = self.est
        S = self._lanes(M)
        iters = est.cfg['refine_iter']
        with torch.no_grad():
            dev_frames = est.detector.upload_frame(frames)
            cams = est.detector._to_dev(glue.cameras(Ks))
            S['cams'].copy_(cams)
            if poses is None:
                pred = est._predict_device_fn(st)

                def fn(frames_, cams_):
                    outs = pred(frames_, cams_)
                    return outs + (self._finish(S, outs[0][-1], True),)
                outs = self.stages.run('start', fn, [dev_frames, cams], state=self._state_list(S))
                out_poses, inter = est._device_results(outs[:-1], M)
                smoothed = self._split(outs[-1], M)[1]
            else:
                f32 = poses.dtype == np.float32

                def fn(frames_, poses_):
                    chain = [poses_]
                    p = poses_
                    for it in range(iters):
                        p = self._refine(st, S, frames_, p, 1, f32 or it > 0)
                        chain.append(p)
                    return torch.stack(chain, 0), self._finish(S, p, True)
                init = est.detector._to_dev(np.ascontiguousarray(poses, np.float64).reshape(M, 12))
                chain, out = self.stages.run(f'start_pose{int(f32)}', fn, [dev_frames, init], state=self._state_list(S))
                chain = est.detector._to_host(chain).reshape(iters + 1, M, 3, 4)
                out_poses, smoothed = self._split(out, M)
                inter = {'refine_poses': [poses] + [c.astype(np.float32) for c in chain[1:]]}
        self._shape = shape
        return out_poses, smoothed, inter

    def step(self, frames, poses=None):
        """Next frames of the M videos: refine_iter refinements from the carried poses (or from `poses` [M,3,4], taken
        as float32, which re-seed the lanes), then smoothing.  Returns (poses float32 [M,3,4], smoothed float64
        [M,3,4] or None)."""
        if self._shape is None:
            raise RuntimeError('Gen6DTracker.step() before start()')
        shape, frames = self._upload(frames)
        if shape != self._shape:
            raise ValueError(f'frames {shape} differ from the started videos {self._shape}')
        M = shape[0]
        if poses is not None and np.shape(poses) != (M, 3, 4):
            raise ValueError(f'poses must be [{M},3,4]')
        st = self._glue()
        est = self.est
        S = self._lanes(M)
        with torch.no_grad():
            dev_frames = est.detector.upload_frame(frames)
            if poses is not None:
                seed = np.asarray(poses).astype(np.float32).astype(np.float64).reshape(M, 12)
                S['poses'].copy_(est.detector._to_dev(seed))

            def fn(frames_):
                return self._finish(S, self._refine(st, S, frames_, S['poses'], self.refine_iter, True), False)
            out = self.stages.run('step', fn, [dev_frames], state=self._state_list(S))
            return self._split(out, M)
