"""Golden vectors of the reference's video tracking loop (predict.py:47-72), produced by the UNMODIFIED reference
estimator on the synthetic in-memory object database and the seeded checkpoints.  Build container only:
    python tests/golden/make_golden_track.py
Outputs tests/golden/track_golden.npz.

The video: 8 frames of SyntheticObjectDatabase.render along a smooth camera path that starts at query view '11'
(track_path() below; the tests render the same frames), with predict.py's pseudo intrinsics f = sqrt(h^2 + w^2).
Frame 0 runs the full prediction (refine_iter = 3), every later frame refine_iter = 1 from the previous pose, and each
pose goes through predict.py's smoothing: project the box of get_ref_point_cloud, weighted_pts (num 5, std 2.5), pnp."""
import importlib.abc
import importlib.machinery
import os
import sys
import tempfile
import types

import numpy as np
import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import ref_shims  # noqa: E402


class _EmptyPackages(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    """matplotlib.* and tqdm as empty packages (every attribute a no-op function): predict.py imports them (through eval.py / utils/draw_utils.py) for
    drawing and progress bars, neither of which the tracking loop below calls."""
    NAMES = ('matplotlib', 'tqdm')

    def find_spec(self, name, path=None, target=None):
        if name.split('.')[0] in self.NAMES:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)
        return None

    def create_module(self, spec):
        m = types.ModuleType(spec.name)
        m.__path__ = []
        m.tqdm = lambda it, *a, **k: it
        m.__getattr__ = lambda attr: (lambda *a, **k: None)      # matplotlib.use('Agg') and the like: no-ops
        return m

    def exec_module(self, module):
        pass


sys.meta_path.insert(0, _EmptyPackages())
ref_shims.install()
import cases  # noqa: E402
import predict as RPR  # noqa: E402  (reference)
from dataset.database import CustomDatabase, get_ref_point_cloud  # noqa: E402  (reference)
from estimator import Gen6DEstimator as RefEstimator  # noqa: E402  (reference)
from utils import base_utils as RB, draw_utils as RDR, pose_utils as RP  # noqa: E402  (reference)

from gen6d_b200.database import SyntheticObjectDatabase  # noqa: E402
from gen6d_b200.network import name2network as ours  # noqa: E402
from gen6d_b200.weights import seeded_state_dict  # noqa: E402
from track_path import track_path  # noqa: E402

torch.set_num_threads(os.cpu_count())
EST = cases.estimator_case()
syn = SyntheticObjectDatabase(**EST['db'])


class RefDB(CustomDatabase):
    """Reference-side view of the synthetic database (as in make_golden_estimator.py)."""

    def __init__(self, s):
        self.database_name = 'custom/synthetic'
        self.s = s
        self.center = s.center
        self.object_point_cloud = s.object_point_cloud
        self.poses, self.Ks, self.img_ids = s.poses, s.Ks, s.img_ids

    def get_image(self, img_id):
        return self.s.get_image(img_id)


db = RefDB(syn)
path, K = track_path(syn)
frames = [syn.render(p, K) for p in path]

work = tempfile.mkdtemp(prefix='g6d_ref_')
os.chdir(work)
cfg = {'name': 'gen6d_synth', 'type': 'gen6d', 'ref_resolution': 128, 'ref_view_num': 64, 'det_ref_view_num': 32,
       'refine_iter': 3}
for name, extra in (('detector', {'vgg_score_stats': cases.DET_STATS_EST}), ('selector', {}), ('refiner', {})):
    sub = {'name': f'{name}_synth', 'network': name, **EST['net_cfg'].get(name, {}), **extra}
    os.makedirs(f'data/model/{sub["name"]}', exist_ok=True)
    torch.save({'network_state_dict': seeded_state_dict(ours[name](sub), cases.WEIGHT_SEED), 'step': 0},
               f'data/model/{sub["name"]}/model_best.pth')
    with open(f'{name}.yaml', 'w') as f:
        yaml.safe_dump(sub, f)
    cfg[name] = f'{name}.yaml'
est = RefEstimator(cfg)
est.build(db, 'all')

# predict.py:36-37, 51-71 (num = 5, std = 2.5: predict.py's argparse defaults)
object_pts = get_ref_point_cloud(db)
bbox = RDR.pts_range_to_bbox_pts(np.max(object_pts, 0), np.min(object_pts, 0))
num, std = 5, 2.5
out = {'track.path': np.stack(path), 'track.K': K, 'track.bbox': bbox, 'track.num': np.asarray(num), 'track.std': np.asarray(std)}
rec = {k: [] for k in ('in_pose', 'pose', 'corners', 'wpts', 'pnp')}
pose_init, hist_pts = None, []
for que_id, img in enumerate(frames):
    if pose_init is not None:
        est.cfg['refine_iter'] = 1
    pose_pr, inter = est.predict(img, K, pose_init=pose_init)
    rec['in_pose'].append(np.asarray(inter['refine_poses'][0], np.float64))
    pose_init = pose_pr
    pts, _ = RB.project_points(bbox, pose_pr, K)
    hist_pts.append(pts)
    pts_ = RPR.weighted_pts(hist_pts, weight_num=num, std_inv=std)
    pose_ = RP.pnp(bbox, pts_, K)
    rec['pose'].append(pose_pr)
    rec['corners'].append(pts)
    rec['wpts'].append(pts_)
    rec['pnp'].append(pose_)
    print('frame', que_id, 'pose', pose_pr.dtype, np.round(pose_pr[:, 3], 4), 'smoothed t', np.round(pose_[:, 3], 4))
for k, v in rec.items():
    out[f'track.{k}'] = np.stack(v)
print({k: (v.dtype, v.shape) for k, v in out.items()})
np.savez_compressed(os.path.join(HERE, 'track_golden.npz'), **out)
print('wrote track_golden.npz')
