"""Tracking throughput of Gen6DTracker on one GPU, against the host-sequenced predict(img, K, pose_init=prev) loop of the
reference's predict.py, measured in the same run.  Prints one JSON line:

  python tools/track_bench.py [--steps 200] [--lanes 1,4,16,32]

For every lane count M (M videos in lockstep, one tracked frame per lane and step):
  * device_fps: tracked frames/s with the frames resident on the device -- replays of the captured step graph only,
    one synchronise at the end;
  * e2e_fps: tracked frames/s end to end -- numpy frames in, numpy poses (+ smoothed poses) out, every step;
  * M = 1 also gives the per-step latency of both.
The baseline is predict(pose_init=prev) with refine_iter = 1 frame after frame (frames/s and per-frame latency), and,
for context, predict_many's poses/s on independent frames.  Every lane count is warmed up before any timing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from golden.track_path import track_path  # noqa: E402
from gen6d_b200.synthetic import build_estimator  # noqa: E402
from gen6d_b200.tracker import Gen6DTracker  # noqa: E402
from oracle.track import bbox_corners  # noqa: E402


def gpu_info():
    """Card name and power limit, read-only, in this run."""
    try:
        out = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(',')[:2]]
        return {'name': name, 'power_limit': power}
    except Exception as exc:            # noqa: BLE001 - reported, not hidden
        return {'name': torch.cuda.get_device_name(0), 'power_limit': f'unavailable ({exc.__class__.__name__})'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--lanes', default='1,4,16,32')
    ap.add_argument('--frames', type=int, default=8, help='distinct video frames per lane, cycled')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('track_bench.py needs a CUDA device')
    lanes = [int(v) for v in args.lanes.split(',')]
    est, db = build_estimator()
    pts = db.object_point_cloud
    bbox = bbox_corners(pts.max(0), pts.min(0)).astype(np.float32)
    Mmax = max(lanes)
    paths, Ks = zip(*[track_path(db, n=args.frames, start=db.get_img_ids()[j % len(db.get_img_ids())]) for j in range(Mmax)])
    frames = [np.stack([db.render(paths[j][k], Ks[j]) for j in range(Mmax)]) for k in range(args.frames)]
    Ks = np.stack(Ks)

    trackers = {}
    for M in lanes:                                     # warm-up: capture start / step graphs of every M
        tr = trackers[M] = Gen6DTracker(est, bbox)
        tr.start(frames[0][:M], Ks[:M])
        for k in range(1, 4):
            tr.step(frames[k][:M])
    torch.cuda.synchronize()

    res = {'gpu': gpu_info(), 'steps': args.steps, 'frame': list(frames[0].shape[1:]), 'lanes': {}}
    for M in lanes:
        tr = trackers[M]
        tr.start(frames[0][:M], Ks[:M])
        step = next(s for k, s in tr.stages.stages.items() if k[0] == 'step')
        tr.step(frames[1][:M])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step.graph.replay()
        torch.cuda.synchronize()
        dev_s = time.perf_counter() - t0
        tr.start(frames[0][:M], Ks[:M])
        t0 = time.perf_counter()
        for s in range(args.steps):
            tr.step(frames[1 + s % (args.frames - 1)][:M])
        e2e_s = time.perf_counter() - t0
        res['lanes'][M] = {'device_fps': round(M * args.steps / dev_s, 1), 'e2e_fps': round(M * args.steps / e2e_s, 1),
                           'device_step_ms': round(1e3 * dev_s / args.steps, 3), 'e2e_step_ms': round(1e3 * e2e_s / args.steps, 3)}

    # today's path: predict(pose_init=prev), refine_iter = 1 after the first frame (predict.py:56-59)
    iters = est.cfg['refine_iter']
    prev, _ = est.predict(frames[0][0], Ks[0])
    est.cfg['refine_iter'] = 1
    try:
        for k in range(1, 4):
            prev, _ = est.predict(frames[k][0], Ks[0], pose_init=prev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(args.steps):
            prev, _ = est.predict(frames[1 + s % (args.frames - 1)][0], Ks[0], pose_init=prev)
        base_s = time.perf_counter() - t0
    finally:
        est.cfg['refine_iter'] = iters
    res['baseline_predict_pose_init'] = {'fps': round(args.steps / base_s, 1), 'frame_ms': round(1e3 * base_s / args.steps, 3)}

    imgs = [frames[k % args.frames][k // args.frames % Mmax] for k in range(64)]
    Kl = [Ks[k // args.frames % Mmax] for k in range(64)]
    est.predict_many(imgs, Kl, workers=2, batch=8)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    est.predict_many(imgs, Kl, workers=2, batch=8)
    res['predict_many_poses_per_s'] = round(64 / (time.perf_counter() - t0), 1)
    base = res['baseline_predict_pose_init']
    res['beats_baseline'] = all(v['device_fps'] > base['fps'] and v['e2e_fps'] > base['fps'] for v in res['lanes'].values()) and \
        res['lanes'].get(1, {'e2e_step_ms': 0})['e2e_step_ms'] < base['frame_ms']
    print(json.dumps(res))


if __name__ == '__main__':
    main()
