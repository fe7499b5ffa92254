"""Contract benchmark: poses/sec of the Gen6D inference hot path (detect -> select -> 3x refine).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pose: a synthetic 480x640 frame through the detector (32 reference views,
4 scales), the 128x128 crop through the selector (64 reference views x 5 in-plane angles), and
three refinement iterations (6 views, 32^3 volume) -- BASELINE.json's full-estimator config.

  value : poses/s of the three-network device path with every input already resident in HBM
          (frame, crop and the three refinement problems were uploaded before the timed region).
  e2e   : poses/s through the public API `Gen6DEstimator.predict(numpy frame, K) -> numpy pose`,
          host geometry (OpenCV warps), pinned H2D copies and D2H reads inside the timed region.
  roofline     : dominant kernel (the implicit-GEMM convolution) timed live with CUDA events.
  cpu_baseline : oracle/ (torch-CPU port of the reference path) timed on the host cores.

N > 1 (torchrun): one process per GPU, each rank runs an independent replica on its own frames
(weak scaling, no data-path collective; poses are all-gathered once at the end over NCCL).
`--impl reference` times the CPU oracle port instead (the reference itself is not part of this
repository).
`--dump-outputs DIR` writes, after the timed steps, what the device-resident path computed for its last
batch and the poses the timed end-to-end call returned (see write_outputs); the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

E2E_WORKERS = int(os.environ.get('G6D_E2E_WORKERS', '2'))      # host threads / CUDA streams per GPU (predict_many / device lanes)
E2E_BATCH = int(os.environ.get('G6D_E2E_BATCH', '0'))          # frames per batched stage (predict_batch); 0 = pick_batch(steps)
E2E_MAX_BATCH = 10


def pick_batch(steps, workers):
    """Frames per batched stage for a timed region of `steps` poses on `workers` lanes: the largest batch <= 10 that
    deals every lane the same number of full batches (steps 20, 2 lanes -> 10; a ragged tail would leave one lane
    idle for a whole batch), 4 when nothing divides.  Measured on B200 at 20 steps (2 lanes): batch 4 -> 164 poses/s
    device-resident / 123-135 end to end, 5 -> 172 / 130, 10 -> 171-174 / 138-142; 1 lane x 20 -> 162 / 139;
    4 lanes x 5 -> 171 / 135."""
    if E2E_BATCH > 0:
        return E2E_BATCH
    if steps % workers == 0:
        per_lane = steps // workers
        for b in range(min(E2E_MAX_BATCH, per_lane), 0, -1):
            if per_lane % b == 0 and (b >= 4 or b == per_lane):
                return b
    return 4 if steps >= 4 * workers else 1      # very short runs: frame by frame (no batch larger than the run)
METRIC = 'poses/sec end-to-end (128^2 crop, 64 refs, 3 refine iters)'
WORKLOAD = ('full estimator detect->select->3x refine: synthetic 480x640 frame, detector 32 refs x 4 scales, '
            'selector 64 refs x 5 angles, refiner 6 views 32^3 volume, seeded random weights')


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the roofline kernels, from the committed
    `ncu --set full` captures of this round (profiles/ncu_traffic.json, written by tools/ncu_summary.py)."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            pass
    return {}


def read_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d.get('bf16_tflops_sustained', d['bf16_tflops']), 'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1400.0, 'src': 'fallback'}


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples taken DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(n)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ---------------------------------------------------------------------------------------------
def usable_cpus():
    from gen6d_b200.geometry import usable_cpus as u
    return u()


def cpu_pose_fn(device='cpu'):
    """Returns (fn, describe): fn() runs ONE network-only pose of the oracle port (a functional torch
    restatement of the reference's three networks) on `device`: 'cpu' = the reference arm / cpu_baseline
    on the host cores; 'cuda' = the same torch ops in eager mode on the B200 (cuDNN / cuBLAS fp32, TF32
    disabled) -- the same-box GPU comparison point BASELINE.md 4.6 asks for."""
    from gen6d_b200 import geometry as G
    from gen6d_b200 import synthetic as syn
    from oracle import gen6d_oracle as O
    torch.set_num_threads(min(usable_cpus(), 64))
    if device != 'cpu':
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
    dv = lambda t: t.to(device)
    sds = {k: {n: dv(v) for n, v in sd.items()} for k, sd in syn.seeded_state_dicts().items()}
    db = syn.synthetic_database()
    g = torch.Generator().manual_seed(5)
    to01 = lambda u8: torch.from_numpy(u8.astype(np.float32) / 255)
    det_refs = dv(torch.rand(32, 3, 128, 128, generator=g))
    sel_refs = dv(torch.rand(5, 64, 3, 128, 128, generator=g))
    ids = db.get_img_ids()[:64]
    poses = dv(torch.from_numpy(np.stack([db.get_pose(i) for i in ids])))
    t0 = time.perf_counter()
    with torch.no_grad():
        det_feats = O.det_load_refs(sds['detector'], det_refs)
        sel_feats, embed = O.sel_load_refs(sds['selector'], sel_refs, poses, dv(torch.zeros(3)), dv(torch.tensor([0., 0., 1.])))
    if device != 'cpu':
        torch.cuda.synchronize()
    load_s = time.perf_counter() - t0
    frame = dv(to01(db.get_image('11')).permute(2, 0, 1)[None].contiguous())
    crop = dv(torch.rand(1, 3, 128, 128, generator=g))
    rq, rr = dv(torch.rand(1, 3, 128, 128, generator=g)), dv(torch.rand(1, 6, 3, 128, 128, generator=g))
    K = dv(torch.tensor([[[304., 0, 64], [0, 304., 64], [0, 0, 1]]]))
    qp = dv(torch.from_numpy(db.get_pose('11'))[None])
    rp = dv(torch.from_numpy(np.stack([db.get_pose(i) for i in ids[:6]]))[None])
    det_cfg = {'vgg_score_stats': syn.DET_SCORE_STATS}

    def one_pose():
        with torch.no_grad():
            o = O.det_detect(sds['detector'], det_cfg, frame, det_feats)
            O.det_parse(o['scores'], o['select_pr_scale'], o['select_pr_offset'])
            lg, ang = O.sel_forward(sds['selector'], crop, sel_feats, embed)
            O.sel_select(lg, ang)
            for _ in range(3):
                O.ref_forward(sds['refiner'], rq, K, qp, rr, K[:, None].repeat(1, 6, 1, 1), rp, 32)

    return one_pose, {'reference_set_load_s': round(load_s, 2)}


def torch_cuda_baseline(steps=10, warm=3):
    """PyTorch eager (cuDNN/cuBLAS fp32, allow_tf32 = False) on the same B200: the oracle port on CUDA
    tensors, device-resident inputs, CUDA events.  A reported comparison point, not a target."""
    fn, info = cpu_pose_fn('cuda')
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {'value': 1e3 / ms, 'unit': 'poses/s', 'ms_per_step': ms, 'steps': steps,
            'what': f'oracle port (functional torch {torch.__version__} restatement of the reference networks) in eager mode on '
                    'cuda:0, cudnn.allow_tf32 = matmul.allow_tf32 = False, one frame at a time, inputs resident, network-only pose'}


def run_torch_cuda_arm(args, rank, world):
    if rank != 0:
        return
    torch.cuda.set_device(0)
    r = torch_cuda_baseline(args.steps, args.warmup)
    print(json.dumps({'impl': 'torch-cuda', 'metric': METRIC, 'value': r['value'], 'unit': 'poses/s', 'n_gpus': 1,
                      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True,
                      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                      'config': {'workload': WORKLOAD, 'path': r['what']}}))


def add_accuracy(est, db):
    """north_star: "at matched ADD-0.1d on synthetic inputs".  The 20 frames of tests/golden/add_golden.npz
    through predict(); ADD-0.1d / Prj-5 against the database's ground truth on the device (g6d_pose_errors),
    next to the values the unmodified reference estimator scored on the same frames (seeded random weights:
    both rates are what an untrained network gives; the check is that they MATCH, frame by frame)."""
    path = os.path.join(ROOT, 'tests', 'golden', 'add_golden.npz')
    if not os.path.exists(path):
        return None
    from gen6d_b200 import metrics as M
    A = np.load(path)
    ids = [str(int(i)) for i in A['frame_ids']]
    poses = np.stack([est.predict(db.get_image(f), db.get_K(f))[0] for f in ids], 0)
    pts, diameter = db.object_point_cloud.astype(np.float32), float(A['diameter'])
    err = M.pose_errors(pts, poses, A['poses_gt'], A['Ks']).cpu().numpy().astype(np.float64)
    return {'frames': len(ids), 'add_0.1d': float(np.mean(err[:, 1] < 0.1 * diameter)), 'prj_5': float(np.mean(err[:, 0] < 5)),
            'reference_add_0.1d': float(A['res.add-0.1d']), 'reference_prj_5': float(A['res.prj-5']),
            'max_abs_add_error_diff_over_0.1d': float(np.abs(err[:, 1] - A['obj_err']).max() / (0.1 * diameter)),
            'max_rel_prj_error_diff': float((np.abs(err[:, 0] - A['prj_err']) / A['prj_err']).max()),
            'reference': 'unmodified reference estimator on CPU, scored by its utils/pose_utils.py (tests/golden/make_golden_add.py)'}


def sharded_section(world, rank, note=lambda what: None):
    """BASELINE configs[3] / [4] on the driver's clock (world > 1): selector with the reference views sharded
    (64 refs x 36 rotation bins per GPU = 2304 slices, 1.585 GB stack per GPU; exact cross-GPU InstanceNorm
    statistics) and refiner with the pose batch sharded (32 poses per GPU, 6 views, 32^3).  CUDA events,
    max over ranks; weak-scaling efficiency = the same per-GPU work run unsharded on this rank / sharded."""
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from golden import cases
    from gen6d_b200 import dist as gdist, ops
    from gen6d_b200.network import name2network
    from gen6d_b200.weights import seeded_state_dict
    comm = gdist.Comm()

    def build(name, cfg):
        net = name2network[name](cfg)
        net.load_state_dict(seeded_state_dict(net, 0))
        return net.cuda().eval()

    def timed(fn, iters, warm=2):
        for _ in range(warm):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / iters], device='cuda', dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    per_gpu_refs, bins, per_gpu_poses = 64, 36, 32
    out = {}
    # ---- selector: references sharded; every rank synthesises the same full set and keeps its slice
    g = torch.Generator().manual_seed(1)
    refs = per_gpu_refs * world
    poses = cases.sphere_poses(3, refs)
    blocks = (torch.rand(bins, refs, 8, 8, 3, generator=g) * 255).to(torch.uint8).numpy()
    imgs = np.repeat(np.repeat(blocks, 16, axis=2), 16, axis=3)          # blocky 128x128 images, same on every rank
    que = cases.rand_images_u8(5, 1, 128, 128, 3)
    center, vert = np.zeros(3, np.float32), np.array([0, 0, 1], np.float32)
    r0, r1 = comm.shard_range(refs)
    note('sharded: inputs synthesised')
    local = build('selector', {'selector_angle_num': bins})
    local.load_ref_imgs(np.ascontiguousarray(imgs[:, r0:r1]), poses[r0:r1], center, vert)
    note('sharded: unsharded selector loaded')
    t_local = timed(lambda: local.select_que_imgs(que), 12, warm=3)
    note('sharded: unsharded selector timed')
    del local
    torch.cuda.empty_cache()
    sel = gdist.shard_selector(build('selector', {'selector_angle_num': bins}), comm)
    sel.load_ref_imgs(imgs, poses, center, vert)
    note('sharded: sharded selector loaded')
    t_shard = timed(lambda: sel.select_que_imgs(que), 12, warm=3)      # 12 queries: one host hiccup no longer moves the mean by 25 %
    note('sharded: sharded selector timed')
    out['selector_ref_shard'] = {
        'workload': f'{refs} refs x {bins} bins over {world} GPUs ({per_gpu_refs} refs = {per_gpu_refs * bins} slices = '
                    f'{per_gpu_refs * bins * 688128 / 1e9:.3f} GB of reference stack per GPU), 1 query 128x128',
        'ms_per_query': t_shard, 'queries_per_s': 1e3 / t_shard, 'ms_per_query_same_shard_unsharded_1gpu': t_local,
        'weak_scaling_efficiency': t_local / t_shard,
        'collectives': sel.comm_stats() if hasattr(sel, 'comm_stats') else None}
    del sel
    torch.cuda.empty_cache()
    # ---- refiner: pose batch sharded
    rfr = build('refiner', {})
    rc = cases.refiner_case(seed=7, qn=per_gpu_poses)        # every rank refines its own 32 poses (same synthetic set)
    dev = lambda x: torch.from_numpy(x).cuda()
    a = [ops.preprocess_u8(dev(rc['que_imgs']), 4, True), dev(rc['que_Ks']), dev(rc['que_poses']),
         ops.preprocess_u8(dev(rc['ref_imgs']), 4, True), dev(rc['ref_Ks']), dev(rc['ref_poses'])]
    note('sharded: refiner inputs ready')
    with torch.no_grad():
        t_one = timed(lambda: rfr._forward_nhwc(*a), 3, warm=1)
        t_all = timed(lambda: comm.all_gather_cat(rfr._forward_nhwc(*a), dim=0), 3, warm=1)
    out['refiner_pose_shard'] = {
        'workload': f'{per_gpu_poses * world} poses over {world} GPUs ({per_gpu_poses} per GPU), 6 views, 32^3 volume, one iteration '
                    '(configs[4] runs 6 of them)',
        'ms_per_iteration': t_all, 'pose_iterations_per_s': per_gpu_poses * world / t_all * 1e3,
        'ms_per_iteration_unsharded_1gpu': t_one, 'weak_scaling_efficiency': t_one / t_all}
    return out


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    fn, info = cpu_pose_fn()
    steps, warm = args.steps, args.warmup
    note = None
    if steps + warm > 40:   # keep the whole run within a few minutes (one CPU pose is ~4-5 s)
        steps = max(1, 40 - warm)
        note = f'steps capped from {args.steps} to {steps} (one CPU pose takes seconds)'
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    dt = time.perf_counter() - t0
    v = steps / dt
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'poses/s', 'n_gpus': args.gpus, 'steps': steps,
            'warmup': warm, 'ms_per_step': dt / steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'path': 'network-only pose (no host warps), torch CPU'},
            'cpu_baseline': {'value': v, 'unit': 'poses/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                             'sample': f'{steps} poses of the oracle port (torch {torch.__version__} CPU kernels)', **info},
            'e2e': {'value': v, 'unit': 'poses/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    if note:
        line['note'] = note
    print(json.dumps(line))


DUMP_LIMIT = 64 << 20           # bytes of .npy files --dump-outputs may write
DUMP_SEED = 0
STAGE_OUTPUTS = {'predict': ('poses', 'detection', 'crop', 'ref_idx', 'selection', 'logits')}   # Gen6DEstimator._predict_device_fn


def stage_outputs(outs):
    """[(stage name, tensor or tuple of tensors)] of one batch -> {'<stage>.<output>': host array}.  A stage name that
    recurs (the per-iteration refine stages of the host-sequenced path) gets its occurrence number appended."""
    names = [n for n, _ in outs]
    seen, res = {}, {}
    for name, o in outs:
        seen[name] = seen.get(name, 0) + 1
        stage = name if names.count(name) == 1 else f'{name}{seen[name] - 1}'
        o = o if isinstance(o, (tuple, list)) else (o,)
        labels = STAGE_OUTPUTS.get(name, ())
        for j, t in enumerate(o):
            res[f'{stage}.{labels[j] if j < len(labels) else j}'] = t.detach().cpu().numpy()
    return res


def write_outputs(path, arrays, limit=DUMP_LIMIT):
    """Writes every array as path/<name>.npy: floating point as float32 (float64 stays float64), integers as float64
    (exact).  An array above its equal share of `limit` is replaced by a fixed, seeded sample of its flattened
    elements, in order.  Returns {name: [shape written, shape computed]}."""
    os.makedirs(path, exist_ok=True)
    share = (limit - 256 * len(arrays)) // max(1, len(arrays))      # 256 bytes of .npy header per file at most
    written = {}
    for name, a in sorted(arrays.items()):
        a = np.asarray(a)
        full = list(a.shape)
        a = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in 'biu' else np.float32)
        if a.nbytes > share:
            keep = np.random.default_rng(DUMP_SEED).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(keep)]
        np.save(os.path.join(path, name + '.npy'), a)
        written[name] = [list(a.shape), full]
    return written


# ---------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    from gen6d_b200 import _lib, graphs, ops
    from gen6d_b200 import geometry as G
    from gen6d_b200 import synthetic as syn
    from gen6d_b200.network import base as nbase

    t_start = time.perf_counter()

    def note(what):         # progress on stderr (rank 0): where the wall-clock of a bench run goes
        if rank == 0:
            print(f'[bench {time.perf_counter() - t_start:6.1f} s] {what}', file=sys.stderr, flush=True)

    torch.cuda.set_device(local_rank)
    ops.require_cuda()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    est, db = syn.build_estimator()
    note('estimator built')
    ids = db.get_img_ids()
    frames = [ids[(7 + rank * 13 + i * 3) % len(ids)] for i in range(8)]   # different frames per rank
    K = db.K

    # ---- stage inputs for the device-resident measurement: every captured stage of one real batched
    # prediction (detect [B frames] -> select [B crops, cut on the device] -> 3 x refine [B x 7 crops]) is
    # recorded with its device-resident inputs and replayed -- exactly what predict_batch launches, minus
    # host geometry and copies.  W lanes (clones with private graphs, shared weights / reference features),
    # each on its own stream, keep W x B frames in flight.
    W, Bt = E2E_WORKERS, pick_batch(args.steps, E2E_WORKERS)
    tail = args.steps % Bt          # poses of the short last batch of the timed region
    batch_imgs = [db.get_image(frames[i % len(frames)]) for i in range(Bt)]

    def record(e, n):
        rec, mods = [], [m for m in (e, e.detector, e.selector, e.refiner) if m is not None]     # e: the whole-prediction graph (device_glue)
        for m in mods:
            def wrapped(name, fn, inputs, _m=m, _o=m.stages.run):
                rec.append((_m, name, fn, list(inputs)))
                return _o(name, fn, inputs)
            m.stages.run = wrapped
        try:
            e.predict_batch(batch_imgs[:n], [K] * n)
        finally:
            for m in mods:
                del m.stages.run
        return rec

    lanes = [torch.cuda.Stream() for _ in range(W)]
    recs, recs_tail = [], []
    for i in range(W):
        e = est if i == 0 else est.worker_clone()
        with torch.cuda.stream(lanes[i]):
            recs.append(record(e, Bt))
            if tail:
                recs_tail.append(record(e, tail))
            lanes[i].synchronize()
    det, sel, rfr = est.detector, est.selector, est.refiner

    def device_batch(i=0, eager=False, short=False):
        """One batch of Bt poses (short=True: of `tail` poses) on lane i through the captured stage graphs (eager=True:
        kernel by kernel).  Returns [(stage name, outputs)] in launch order."""
        outs = []
        with torch.no_grad():
            for m, name, fn, inputs in (recs_tail if short else recs)[0 if eager else i % W]:
                outs.append((name, fn(*inputs) if eager else m.stages.run(name, fn, inputs)))
        return outs

    last_outputs = []

    def device_steps(n):
        """n poses = n // Bt full batches and, for n % Bt == tail, one short batch, dealt round-robin to the lanes."""
        nb, short = divmod(n, Bt)
        assert short in (0, tail), (n, Bt, tail)
        main = torch.cuda.current_stream()
        for st in lanes:
            st.wait_stream(main)
        for i in range(nb + (short > 0)):
            with torch.cuda.stream(lanes[i % W]):
                last_outputs[:] = device_batch(i, short=i == nb)
        for st in lanes:
            main.wait_stream(st)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warm, takes_index=False, batched=False):
        if batched:
            fn(warm)
        else:
            for _ in range(warm):
                fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count() + graphs.REPLAYED_KERNELS[0]
        w0 = time.perf_counter()
        e0.record()
        if batched:
            fn(steps)
        else:
            for i in range(steps):
                fn(i) if takes_index else fn()
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - w0
        ms = max(e0.elapsed_time(e1), 0.0)
        launches = _lib.launch_count() + graphs.REPLAYED_KERNELS[0] - l0
        barrier()
        t = torch.tensor([ms, wall * 1e3], device='cuda', dtype=torch.float64)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), launches

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    note('stage graphs recorded')
    dev_ms, _, launches = timed(device_steps, args.steps, -(-max(args.warmup, 2 * W * Bt) // Bt) * Bt, batched=True)
    dumps = stage_outputs(last_outputs) if args.dump_outputs else {}

    note('device-resident timing done')
    # ---- end to end through the public API (numpy in, numpy out)
    imgs = [db.get_image(f) for f in frames]
    nbase.IO_BYTES['h2d'] = nbase.IO_BYTES['d2h'] = 0
    out_poses = []

    def e2e_step(i=0):
        pose, _ = est.predict(imgs[i % len(imgs)], K)
        out_poses.append(pose)

    _, e2e_wall_ms, _ = timed(e2e_step, args.steps, args.warmup, takes_index=True)
    io = dict(nbase.IO_BYTES)
    n_calls = args.steps + args.warmup

    note('single-frame e2e done')
    # the throughput API: W host threads x batches of Bt frames through predict_batch
    def pipelined(n):
        res = est.predict_many([imgs[i % len(imgs)] for i in range(n)], [K] * n, workers=E2E_WORKERS, batch=Bt)
        out_poses.extend(r[0] for r in res)

    pipelined(2 * E2E_WORKERS * Bt)             # builds the worker clones, captures their graphs
    pipelined(max(args.warmup, E2E_WORKERS * Bt))   # untimed warm-up of the whole pipelined path
    barrier()
    t0 = time.perf_counter()
    pipelined(args.steps)
    torch.cuda.synchronize()
    pipe_ms = (time.perf_counter() - t0) * 1e3
    if args.dump_outputs:
        dumps['e2e.poses'] = np.stack(out_poses[-args.steps:], 0)
    barrier()
    if world > 1:
        import torch.distributed as dist
        tt = torch.tensor([pipe_ms], device='cuda', dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        pipe_ms = float(tt[0])
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        import torch.distributed as dist
        mine = torch.from_numpy(np.stack(out_poses[-args.steps:], 0)).cuda()
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)       # the only collective: results, once, at the end

    note('pipelined e2e done')
    # ---- live kernel timing (CUDA events around every launch of the three kernels of interest)
    os.environ['G6D_BRANCH_STREAMS'] = '0'      # per-kernel timing: one kernel at a time, no co-scheduling
    device_batch(0, eager=True)
    torch.cuda.synchronize()
    prof = ops.enable_profiling()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    device_batch(0, eager=True)
    pe1.record()
    torch.cuda.synchronize()
    eager_ms = pe0.elapsed_time(pe1)
    stats = ops.collect_profile(prof)
    os.environ.pop('G6D_BRANCH_STREAMS', None)
    peaks = read_peaks()
    conv = stats.get('g6d_conv_tc', {'ms': 0, 'work': 0, 'n': 1})
    ffma = stats.get('g6d_conv', {'ms': 0, 'work': 0, 'n': 0})
    f16 = ops.conv_kind() == _lib.TC_F16
    split = 3.0 if f16 else 6.0             # bf16-peak units per fp32-equivalent flop: 3 fp16 MMAs, or 3 TF32 MMAs at half rate
    traffic = ncu_traffic()
    roof = {'kernel': 'conv_tc2_kernel / conv_tcflat_kernel (tcgen05 implicit-GEMM convolution, fp32-faithful 3-term operand split, '
                      + ('fp16 hi + 2^11-scaled fp16 lo halves, kind::f16' if f16 else 'tf32 hi/lo halves, kind::tf32') + ')',
            'bound': 'tensor', 'achieved': conv['work'] / max(conv['ms'], 1e-9) / 1e9, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
            'traffic': traffic.get('conv'),
            'traffic_of': 'DRAM bytes of ONE launch of the 3x3 512->512 layer on a 120x160 map (tools/conv_one.py, ncu --set full): '
                          'its 4.2 GB of operand reads are served from L2; activations + weights come from HBM once',
            'peak_source': f"{peaks['src']} bf16 dense GEMM (sustained); achieved counts fp32-equivalent flops 2MNK, each issued as 3 "
                           + ('fp16' if f16 else 'TF32') + f" MMAs, so 1/{split:g} of this peak is the ceiling of the parity mode",
            'launches_per_step': conv['n'] / Bt, 'ms_per_step': conv['ms'] / Bt,
            'share_of_step': conv['ms'] / max(eager_ms, 1e-9),
            'timing': f'CUDA events around every launch in an extra serialised pass (branch streams off, one batch of {Bt} frames, kernel by '
                      'kernel): ms_per_step here is un-overlapped kernel time per pose and exceeds the top-level ms_per_step, which overlaps '
                      'lanes and branches',
            'ffma_fallback': {'launches_per_step': ffma['n'] / Bt, 'ms_per_step': ffma['ms'] / Bt,
                              'tflops': ffma['work'] / max(ffma['ms'], 1e-9) / 1e9}}
    roof['frac'] = roof['achieved'] / roof['peak']
    roof['frac_of_split_ceiling'] = roof['achieved'] / (roof['peak'] / split)
    roof['frac_of_3xtf32_ceiling'] = roof['achieved'] / (roof['peak'] / 6.0)     # round-1 yardstick, kept for continuity
    extra = []
    for key, label, units in (('g6d_sel_corr_score3', 'selector correlation + rotated-similarity score, 3 levels (S2)', 1),
                              ('g6d_ref_volume_fill', 'refiner unproject-and-aggregate volume fill (R2)', Bt)):
        if key in stats:
            s = stats[key]
            ach = s['work'] / max(s['ms'], 1e-9) / 1e6
            extra.append({'kernel': label, 'bound': 'hbm', 'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                          'frac': ach / peaks['hbm_gbs'], 'us_per_launch': s['ms'] / s['n'] * 1e3,
                          'units_per_launch': units, 'unit_is': 'one query' if units == 1 else 'one pose-iteration (the batched refine stage fills all volumes of the batch in one launch)',
                          'algorithmic_bytes_per_unit': s['work'] / s['n'] / units,
                          'traffic': traffic.get('s2' if 'score3' in key else 'r2'),
                          'traffic_of': 'dram__bytes_read.sum + dram__bytes_write.sum of one launch with ONE unit (ncu --set full on tools/profile_step.py)'
                                        + ('' if units == 1 else '; the 50 MB the kernel writes per unit stay in L2 for the embed convolutions that read them next')})
    note('kernel timing done')
    accuracy = add_accuracy(est, db) if rank == 0 else None
    note('accuracy done')
    sharded = sharded_section(world, rank, note) if world > 1 else None
    note('sharded section done')
    if rank != 0:
        return
    value = world * args.steps / (dev_ms * 1e-3)
    e2e_v = world * args.steps / (e2e_wall_ms * 1e-3)
    line = {'metric': METRIC, 'value': value, 'unit': 'poses/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'parallelism': f'replica x{world} (independent frames per GPU); per GPU {E2E_WORKERS} lanes (streams) x batches of '
                                                            f'{Bt} frames through the batched stages = {E2E_WORKERS * Bt} frames in flight' + ('; camera algebra between the stages on the device, one captured graph per batch' if est.cfg['device_glue'] else '; stages sequenced by the host'),
                       'l2': 'per-step working set (220 MB selector reference stack + 300 MB weights + detector '
                             'activations) exceeds the 126 MB L2; no explicit flush'},
            'e2e': {'value': world * args.steps / (pipe_ms * 1e-3), 'unit': 'poses/s', 'ms_per_step': pipe_ms / args.steps,
                    'h2d_bytes_per_step': io['h2d'] // n_calls, 'd2h_bytes_per_step': io['d2h'] // n_calls,
                    'api': f'Gen6DEstimator.predict_many(numpy frames, Ks, workers={E2E_WORKERS}, batch={Bt}) -> numpy poses: {E2E_WORKERS} host threads '
                           f'each push batches of {Bt} frames through predict_batch (pinned H2D of the frames once, crops cut from them on the device, '
                           'camera geometry on the host, one D2H per stage and batch)',
                    'single_frame_latency': {'value': e2e_v, 'unit': 'poses/s', 'ms_per_step': e2e_wall_ms / args.steps,
                                             'api': 'Gen6DEstimator.predict(numpy frame, K), one frame at a time'}},
            'gpu_launches': int(launches), 'roofline': roof, 'kernels': extra, 'clocks': clocks}
    if accuracy is not None:
        line['accuracy'] = accuracy
    if sharded is not None:
        line['sharded'] = sharded
    if args.dump_outputs:
        line['dumped_outputs'] = write_outputs(args.dump_outputs, dumps)
    if world == 1:
        try:
            line['torch_cuda_baseline'] = torch_cuda_baseline(5, 2)
        except Exception as e:  # noqa: BLE001  (a reported comparison point must not take the bench line down)
            line['torch_cuda_baseline'] = {'unavailable': repr(e)[:200]}
        fn, info = cpu_pose_fn()        # sets torch threads to the usable-CPU count for the CPU baseline
        fn()
        n = 2
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        dt = time.perf_counter() - t0
        line['cpu_baseline'] = {'value': n / dt, 'unit': 'poses/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                                'sample': f'{n} network-only poses of the oracle port after 1 warm-up '
                                          f'(torch {torch.__version__} CPU kernels)', **info}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=None)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'torch-cuda'])
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the timed device-resident path computed in its last batch, and the poses of the timed '
                         'end-to-end call, as DIR/<name>.npy (float32 / float64, at most 64 MB in all)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        args.steps = 5 if args.steps is None else args.steps
        args.warmup = 1 if args.warmup is None else args.warmup
        run_reference_arm(args, rank, world)
        return
    if args.impl == 'torch-cuda':
        args.steps = 10 if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else max(3, args.warmup)
        run_torch_cuda_arm(args, rank, world)
        return
    args.steps = 20 if args.steps is None else args.steps
    args.warmup = 3 if args.warmup is None else max(3, args.warmup)
    run_ours(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
