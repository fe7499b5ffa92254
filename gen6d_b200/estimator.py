"""Gen6DEstimator on the B200 networks: same constructor / build / predict contract as the
reference's estimator.py:94-216 (numpy images and poses in, numpy pose out; `ref_info`, `cfg`).

The stage sequencing is inherently serial per frame (crop depends on the detection, refinement
k+1 on pose k), so this class keeps the reference's structure; throughput comes from the kernels,
from keeping every reference-side tensor resident on the device, and from running independent
frames on independent GPUs (see gen6d_b200/dist.py).
"""
import os

import numpy as np
import torch
import yaml

from . import geometry as G
from . import glue
from . import ops
from .graphs import StageCache
from .network import name2network


class Gen6DEstimator:
    default_cfg = {
        'ref_resolution': 128,
        'ref_view_num': 64,
        'det_ref_view_num': 32,
        'selector': None,
        'detector': None,
        'refiner': None,
        'refine_iter': 3,
        'device_build': False,    # True: cut the 64 + 5x64 reference crops of build() with the device warp kernel (row f2)
        'host_warps': False,      # True: keep the between-stage crops on the host in OpenCV, as the reference does
        'host_threads': None,     # OpenCV / torch-CPU threads for the host geometry (None: min(8, usable CPUs))
        # predict_batch / predict_many(batch > 1) keep the camera algebra between the stages on the device: the whole
        # batch prediction is ONE captured graph (csrc/glue.cu), no host round trips.  False (or G6D_DEVICE_GLUE=0):
        # the host sequences the stages with numpy geometry in between, as predict() does.
        'device_glue': os.environ.get('G6D_DEVICE_GLUE', '1') != '0',
    }

    def __init__(self, cfg, modules=None):
        """cfg: the reference's estimator yaml as a dict (configs/gen6d_pretrain.yaml).  `modules`
        optionally injects already-built networks {'detector','selector','refiner'} (used with
        synthetic checkpoints); otherwise they are loaded like estimator.py:117-125 does."""
        self.cfg = {**self.default_cfg, **cfg}
        self.ref_info = {}
        self.stages = StageCache()        # whole-prediction graphs of the device-glue path
        self._glue = None
        G.configure_host_threads(self.cfg['host_threads'])
        if modules is not None:
            self.detector, self.selector = modules['detector'], modules['selector']
            self.refiner = modules.get('refiner')
        else:
            self.detector = self._load_module(self.cfg['detector'])
            self.selector = self._load_module(self.cfg['selector'])
            self.refiner = self._load_module(self.cfg['refiner']) if self.cfg['refiner'] is not None else None

    @staticmethod
    def _load_module(cfg_path):
        with open(cfg_path, 'r') as f:
            cfg = yaml.load(f, Loader=yaml.FullLoader)
        net = name2network[cfg['network']](cfg)
        state = torch.load(f'data/model/{cfg["name"]}/model_best.pth', map_location='cpu')
        net.load_state_dict(state['network_state_dict'])
        print(f'load from {cfg["name"]}/model_best.pth step {state["step"]}')
        return net.cuda().eval()

    def build(self, database, split_type='all'):
        """estimator.py:139-171: pick 64 well-spread reference views, normalise them to 128x128
        look-at crops, make the 5 in-plane rotated copies, and load the three networks."""
        if split_type != 'all':
            raise NotImplementedError("only the 'all' split (reference ids = all database ids) is supported")
        from .database import as_object_database
        database = as_object_database(database)       # reference-repo databases are wrapped on the fly
        self._drop_workers()                           # clones made for a previous object are stale now
        center, vert = database.object_center(), database.object_vert()
        ids_all = database.get_img_ids()
        ref_ids = G.select_views_fps(database, ids_all, self.cfg['ref_view_num'])
        res = self.cfg['ref_resolution']
        on_device = self.cfg['device_build']
        ref_imgs, ref_Ks, ref_poses, ref_Hs = G.normalize_reference_views(database, ref_ids, res, 0.05, warp=not on_device)
        rot_Hs = [[G.similarity_2d((res / 2, res / 2), 1.0, ang, (res / 2, res / 2)).astype(np.float32) @ ref_Hs[k]
                   for k in range(len(ref_ids))] for ang in (-np.pi / 2, -np.pi / 4, 0, np.pi / 4, np.pi / 2)]
        if on_device:
            # same bytes as the OpenCV path (g6d_warp_perspective_u8 is bit-exact), one launch per set
            srcs = [torch.from_numpy(np.ascontiguousarray(database.get_image(i))).to(self.detector.device) for i in ref_ids]
            cut = lambda Hs: ops.warp_perspective_u8(
                torch.from_numpy(G.pack_warp_jobs(srcs, [G.perspective_dst_to_src(H) for H in Hs])).to(srcs[0].device),
                len(srcs), res, res).cpu().numpy()
            ref_imgs = cut(list(ref_Hs))
            rots = [cut(Hs) for Hs in rot_Hs]
        else:
            import cv2
            rots = [np.stack([cv2.warpPerspective(database.get_image(i), Hs[k], (res, res), flags=cv2.INTER_LINEAR)
                              for k, i in enumerate(ref_ids)], 0) for Hs in rot_Hs]
        ref_imgs_rots = np.stack(rots, 0)  # an,rfn,h,w,3
        self.detector.load_ref_imgs(ref_imgs[:self.cfg['det_ref_view_num']])
        self.selector.load_ref_imgs(ref_imgs_rots, ref_poses, center, vert)
        self.ref_info = {'imgs': ref_imgs, 'ref_imgs': ref_imgs_rots, 'Ks': ref_Ks, 'poses': ref_poses,
                         'center': center, 'ref_ids': ref_ids}
        if self.refiner is not None:
            self.refiner.load_ref_imgs(database, ids_all)
        torch.cuda.current_stream().synchronize()      # reference state complete before any other stream reads it

    def predict(self, que_img, que_K, pose_init=None):
        """estimator.py:173-216.  que_img uint8 [h,w,3], que_K [3,3] -> (pose [3,4], inter_results)."""
        inter = {}
        res = self.cfg['ref_resolution']
        host_warps = self.cfg['host_warps']
        # the frame goes to the device once; the detection crop and the refinement look-at crops are
        # cut from it there (bit-exact with the OpenCV warps the reference runs on the host)
        frame = None if host_warps else self.detector.upload_frame(que_img)
        if pose_init is None:
            det = self.detector.detect_que_imgs(que_img[None], que_dev=None if host_warps else frame[None])
            position, scale_r2q = det['positions'][0], det['scales'][0]
            if host_warps:
                crop, _ = G.crop_similarity(que_img, position, 1 / scale_r2q, 0, res)
                sel = self.selector.select_que_imgs(crop[None])
            else:
                _, M = G.crop_similarity(None, position, 1 / scale_r2q, 0, res)
                sel = self.selector.select_from_frame(frame, M, res)
                crop = sel['que_imgs'][0]
            inter.update(det_position=position, det_scale_r2q=scale_r2q, det_que_img=crop)
            ref_idx, angle_r2q, scores = sel['ref_idx'][0], sel['angles'][0], sel['scores'][0]
            inter.update(sel_angle_r2q=angle_r2q, sel_scores=scores, sel_ref_idx=ref_idx)
            pose = G.pose_from_similarity(position, scale_r2q, angle_r2q, self.ref_info['poses'][ref_idx],
                                          self.ref_info['Ks'][ref_idx], que_K, self.ref_info['center'])
        else:
            pose = pose_init
        if self.refiner is not None:
            poses = [pose]
            for _ in range(self.cfg['refine_iter']):
                pose = self.refiner.refine_que_imgs(que_img, que_K, pose, size=128, ref_num=6, ref_even=True,
                                                    que_dev=frame, host_warps=host_warps)
                poses.append(pose)
            inter['refine_poses'] = poses
        return pose, inter


    def predict_batch(self, que_imgs, que_Ks, pose_inits=None):
        """predict() for a batch of independent frames of one size (row f3): qn frames go through ONE
        detect stage, ONE select stage and ONE refine stage per iteration -- 2 + refine_iter graph launches
        and device->host reads for the whole batch instead of per frame -- with the small per-frame camera
        algebra on the host in between.  Same results as predict() frame by frame.
        que_imgs: list / array of uint8 [h,w,3]; que_Ks: [qn,3,3].  Returns (poses [qn,3,4], inter dict of lists)."""
        qn, res = len(que_imgs), self.cfg['ref_resolution']
        que_Ks = [np.asarray(K) for K in que_Ks]
        frames = self.detector.upload_frame([np.asarray(f) for f in que_imgs])  # [qn,h,w,3] once, for all stages
        if self.cfg['device_glue'] and pose_inits is None and self._glue_possible():
            return self._predict_batch_device(frames, que_Ks)
        inter = {}
        if pose_inits is None:
            det = self.detector.detect_que_imgs(None, que_dev=frames)
            Ms = [G.crop_similarity(None, det['positions'][i], 1 / det['scales'][i], 0, res)[1] for i in range(qn)]
            sel = self.selector.select_from_frames(frames, Ms, res)
            inter.update(det_position=det['positions'], det_scale_r2q=det['scales'], det_que_img=sel['que_imgs'],
                         sel_angle_r2q=sel['angles'], sel_scores=sel['scores'], sel_ref_idx=sel['ref_idx'])
            ridx = np.asarray(sel['ref_idx'])
            poses = G.poses_from_similarity(det['positions'], det['scales'], sel['angles'], self.ref_info['poses'][ridx],
                                            self.ref_info['Ks'][ridx], np.stack(que_Ks, 0), self.ref_info['center'])
        else:
            poses = np.stack(pose_inits, 0)
        if self.refiner is not None:
            chain = [poses]
            for _ in range(self.cfg['refine_iter']):
                poses = self.refiner.refine_batch(frames, que_Ks, poses, size=128, ref_num=6, ref_even=True)
                chain.append(poses)
            inter['refine_poses'] = chain
        return poses, inter

    # ------------------------------------------------------------------ device-resident prediction
    def _glue_possible(self):
        return self.refiner is not None and getattr(self.selector.comm, 'capturable', False) and not self.cfg['host_warps']

    def _glue_state(self):
        """Device tables of the camera algebra (glue.py), rebuilt when any module's state changed."""
        gen = self._generation()
        if self._glue is None or self._glue['gen'] != gen:
            dev = self.detector.device
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
            refs = glue.selector_refs(self.ref_info)
            refs_dev = {k: up(refs[k]) for k in ('poses', 'cen', 'f', 'dist')}
            tables = glue.refiner_views(self.refiner.ref_database, self.refiner.ref_ids, 128, 6)
            src = self.refiner._ref_sources(self.refiner.ref_ids)
            views_dev = {k: up(tables[k]) for k in ('poses', 'R_look', 'RlookR', 'f', 'Kinv', 'even_idx', 'even_dirs')}
            views_dev['src'] = up(np.asarray([s[0] for s in src], np.uint64).view(np.int64))
            views_dev['rows'], views_dev['cols'] = up(np.asarray([s[1] for s in src], np.int32)), up(np.asarray([s[2] for s in src], np.int32))
            torch.cuda.current_stream().synchronize()
            ptr = lambda d: {k: t.data_ptr() for k, t in d.items()}
            self._glue = {'gen': gen, 'keep': (refs_dev, views_dev), 'tables': tables,
                          'refs': glue.refs_struct({**ptr(refs_dev), 'center': refs['center']}),
                          'views': glue.views_struct(ptr(views_dev), tables, views_dev['src'].data_ptr(), views_dev['rows'].data_ptr(),
                                                     views_dev['cols'].data_ptr())}
            self.stages.clear()
        return self._glue

    def _predict_device_fn(self, st):
        """frames u8 [qn,h,w,3], cams f64 [qn,20] -> every stage of predict_batch, enqueued back to back."""
        res, iters, R = self.cfg['ref_resolution'], self.cfg['refine_iter'], st['tables']['ref_num']
        select, refine = self.selector._select_warped(res), self.refiner._refine_warped(128)

        def fn(frames, cams):
            det = self.detector._detect_u8(frames)                                  # [qn,4]: x, y, scale, score
            crop, idx, sel_out, logits = select(ops.glue_detection_jobs(det, frames, res))
            poses = ops.glue_initial_poses(det, idx, sel_out, st['refs'], cams)
            chain = [poses]
            for it in range(iters):
                jobs, que_K, que_pose, rect, ref_Ks, ref_poses, _ = ops.glue_refine_problems(st['views'], R, cams, frames, poses, it > 0)
                out = refine(jobs, que_K, que_pose, ref_Ks, ref_poses)
                poses = ops.glue_apply_refinements(st['views'], que_pose, que_K, rect, out)
                chain.append(poses)
            return torch.stack(chain, 0), det, crop, idx, sel_out, logits
        return fn

    def _predict_batch_device(self, frames, que_Ks):
        """predict_batch with cfg['device_glue']: one graph launch, one synchronising read at the end."""
        st = self._glue_state()
        qn = frames.shape[0]
        with torch.no_grad():
            cams = self.detector._to_dev(glue.cameras(np.stack(que_Ks, 0)))
            outs = self.stages.run('predict', self._predict_device_fn(st), [frames, cams])
            return self._device_results(outs, qn)

    def _device_results(self, outs, qn):
        """_predict_device_fn's outputs -> predict_batch's (poses, inter), read back to the host."""
        chain, det, crop, idx, sel_out, logits = [self.detector._to_host(t) for t in outs]
        chain = chain.reshape(len(chain), qn, 3, 4)
        poses0, refined = chain[0], [c.astype(np.float32) for c in chain[1:]]
        inter = {'det_position': det[:, :2].copy(), 'det_scale_r2q': det[:, 2].copy(), 'det_que_img': crop,
                 'sel_angle_r2q': sel_out[:, 0].copy(), 'sel_scores': logits, 'sel_ref_idx': idx,
                 'refine_poses': [poses0] + refined}
        return (refined[-1] if refined else poses0), inter

    # ------------------------------------------------------------------ throughput API
    def worker_clone(self):
        import copy
        other = copy.copy(self)
        other._workers, other._pool, other._workers_gen = None, None, None
        other.stages = StageCache()                   # private graphs; the glue tables (self._glue) are shared, read-only
        other.detector, other.selector = self.detector.worker_clone(), self.selector.worker_clone()
        other.refiner = self.refiner.worker_clone() if self.refiner is not None else None
        return other

    def _generation(self):
        mods = (self.detector, self.selector, self.refiner)
        return tuple(m.generation for m in mods if m is not None)

    def _drop_workers(self):
        pool = getattr(self, '_pool', None)
        if pool is not None:
            pool.shutdown(wait=True)
        self._workers, self._pool, self._workers_gen, self._warm = None, None, None, set()

    def predict_many(self, que_imgs, que_Ks, workers=2, batch=1):
        """Poses for independent frames: `workers` host threads, each with a clone of the networks (shared
        weights / reference features, private CUDA graphs) and a CUDA stream, each pushing `batch` frames
        at a time through predict_batch (batch = 1: plain predict), so one batch's host geometry overlaps
        another batch's kernels.  Same results as predict(); returns [(pose, inter)] (inter of a batched
        frame holds that frame's slices)."""
        from concurrent.futures import ThreadPoolExecutor
        if len(que_imgs) == 0:
            return []
        # The clones share weights / reference features by reference and own captured graphs over them:
        # rebuild them whenever any module's state changed (build() on another object, load_state_dict).
        if getattr(self, '_workers', None) is None or len(self._workers) != workers or self._workers_gen != self._generation():
            self._drop_workers()
            self._workers = [(self.worker_clone(), torch.cuda.Stream()) for _ in range(workers)]
            self._workers_gen = self._generation()
            self._pool = ThreadPoolExecutor(workers)
            self._warm = set()
        n = len(que_imgs)
        batch = max(1, min(batch, n))
        warm_key = (batch, bool(self.cfg['device_glue']))
        if warm_key not in self._warm:               # capture every worker's graphs for this batch size / path, one at a time
            for est, stream in self._workers:
                stream.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(stream):
                    if batch == 1:
                        est.predict(que_imgs[0], que_Ks[0])
                    else:
                        est.predict_batch([que_imgs[i % n] for i in range(batch)], [que_Ks[i % n] for i in range(batch)])
                    stream.synchronize()
            self._warm.add(warm_key)
        results = [None] * n
        caller = torch.cuda.current_stream()
        chunks = [list(range(b, min(b + batch, n))) for b in range(0, n, batch)]

        def run(w):
            est, stream = self._workers[w]
            stream.wait_stream(caller)               # order after whatever the caller enqueued (uploads, a rebuild)
            with torch.cuda.stream(stream):
                for c in range(w, len(chunks), workers):
                    idx = chunks[c]
                    if batch == 1:
                        results[idx[0]] = est.predict(que_imgs[idx[0]], que_Ks[idx[0]])
                        continue
                    pad = idx + [idx[-1]] * (batch - len(idx))        # a short last chunk reuses the captured batch size
                    poses, inter = est.predict_batch([que_imgs[i] for i in pad], [que_Ks[i] for i in pad])
                    for j, i in enumerate(idx):
                        one = {k: ([p[j] for p in v] if k == 'refine_poses' else v[j]) for k, v in inter.items()}
                        results[i] = (poses[j], one)
                stream.synchronize()

        import sys
        old_si = sys.getswitchinterval()
        sys.setswitchinterval(2e-4)      # a worker that just got its D2H result should not wait 5 ms for the GIL
        try:
            list(self._pool.map(run, range(workers)))
        finally:
            sys.setswitchinterval(old_si)
        return results


name2estimator = {'gen6d': Gen6DEstimator}
