"""The viewpoint selector's select stage alone, as the flagship path runs it: crops already on the device, the stage
(preprocess -> VGG -> correlation score -> towers -> tail -> parse) captured as one CUDA graph per batch size and
replayed, timed with CUDA events.  Prints one JSON line:

  python tools/select_bench.py [--qn 1,4,10] [--iters 50]

For every batch size qn: ms per replay, ms per query, and the kernels captured in the stage (launches per stage).
The selector is the estimator's (bench.py's synthetic object: 64 references x 5 in-plane angles, 128x128 crops);
the crops are seeded noise.  Only the selector's long-standing entry points are used (_select_u8 on a uint8 batch),
so the same script measures any revision of the library.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gen6d_b200.graphs import CapturedStage  # noqa: E402
from gen6d_b200.synthetic import build_estimator  # noqa: E402


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
    ap.add_argument('--qn', default='1,4,10')
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--repeats', type=int, default=5, help='timed windows per batch size; the median is reported')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('select_bench.py needs a CUDA device')
    est, _ = build_estimator()
    sel = est.selector
    res = est.cfg['ref_resolution']
    rfn, an = sel.ref_shape
    gen = torch.Generator().manual_seed(0)
    out = {'metric': 'select_stage', 'gpu': gpu_info(), 'refs': rfn, 'angles': an, 'crop': res, 'iters': args.iters, 'qn': {}}
    stages = {}
    for qn in [int(v) for v in args.qn.split(',')]:       # capture (and warm up) every size before timing any
        crops = torch.randint(0, 256, (qn, res, res, 3), generator=gen, dtype=torch.uint8).cuda()
        stages[qn] = (CapturedStage(sel._select_u8, [crops]), crops)
    for qn, (st, crops) in stages.items():
        for _ in range(5):
            st(crops)
        times = []
        for _ in range(args.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                st.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / args.iters)
        ms = sorted(times)[len(times) // 2]
        out['qn'][str(qn)] = {'ms_per_stage': round(ms, 4), 'ms_per_query': round(ms / qn, 4),
                              'spread_ms': round(max(times) - min(times), 4), 'launches_per_stage': st.kernels}
    print(json.dumps(out))


if __name__ == '__main__':
    main()
