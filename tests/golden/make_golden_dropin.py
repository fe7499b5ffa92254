"""Golden data for tests/test_dropin.py from the UNMODIFIED reference (network/, estimator.py and
dataset/database.py, imported through ref_shims).  Build container only:
    python tests/golden/make_golden_dropin.py
Outputs tests/golden/dropin_golden.json:
  * signatures    : parameter names and defaults of every network method the reference estimator calls;
  * estimator_imports / estimator_calls : what estimator.py takes from `network` and which methods it calls
                    on self.detector / self.selector / self.refiner (read from its syntax tree);
  * database      : what the reference's free functions get_object_center / get_diameter / get_object_vert
                    return for a CustomDatabase over SyntheticObjectDatabase(n_views=12, 120x160, seed=3)."""
import ast
import inspect
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import ref_shims  # noqa: E402

ref_shims.install(networks=True)
import network as ref_network  # noqa: E402  (reference)
from dataset.database import CustomDatabase, get_diameter, get_object_center, get_object_vert  # noqa: E402  (reference)
from gen6d_b200.database import SyntheticObjectDatabase  # noqa: E402

NETS = ('detector', 'selector', 'refiner')
METHODS = {'detector': ('__init__', 'load_ref_imgs', 'detect_que_imgs', 'forward'),
           'selector': ('__init__', 'load_ref_imgs', 'select_que_imgs', 'forward'),
           'refiner': ('__init__', 'load_ref_imgs', 'refine_que_imgs', 'forward')}

out = {'signatures': {}, 'estimator_imports': [], 'estimator_calls': {n: [] for n in NETS}}
for name, methods in METHODS.items():
    out['signatures'][name] = {}
    for m in methods:
        params = inspect.signature(getattr(ref_network.name2network[name], m)).parameters.values()
        out['signatures'][name][m] = [[p.name, p.default is not inspect.Parameter.empty,
                                       None if p.default is inspect.Parameter.empty else p.default] for p in params]

tree = ast.parse(open(os.path.join(ref_shims.REFERENCE_ROOT, 'estimator.py')).read())
for node in ast.walk(tree):
    if isinstance(node, ast.ImportFrom) and node.module == 'network':
        out['estimator_imports'] += [a.name for a in node.names]
    # self.<net>.<method>(...)
    if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and isinstance(node.func.value, ast.Attribute)
            and isinstance(node.func.value.value, ast.Name) and node.func.value.value.id == 'self'
            and node.func.value.attr in NETS):
        out['estimator_calls'][node.func.value.attr].append(node.func.attr)
out['estimator_calls'] = {k: sorted(set(v)) for k, v in out['estimator_calls'].items()}


class RefDB(CustomDatabase):
    def __init__(self, s):      # CustomDatabase.__init__ reads a COLMAP project from disk: set its attributes directly
        self.database_name = 'custom/synthetic'
        self.s, self.center, self.object_point_cloud = s, s.center, s.object_point_cloud
        self.poses, self.Ks, self.img_ids = s.poses, s.Ks, s.img_ids


rdb = RefDB(SyntheticObjectDatabase(n_views=12, height=120, width=160, seed=3))
enc = lambda a: {'value': np.asarray(a).tolist(), 'dtype': str(np.asarray(a).dtype)}
out['database'] = {'object_center': enc(get_object_center(rdb)), 'diameter': enc(get_diameter(rdb)),
                   'object_vert': enc(get_object_vert(rdb))}

with open(os.path.join(HERE, 'dropin_golden.json'), 'w') as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write('\n')
print(json.dumps(out, sort_keys=True))
