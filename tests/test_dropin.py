"""The upper face of the drop-in boundary (SURVEY.md 8b), checked against what the UNMODIFIED reference
declares and computes (tests/golden/dropin_golden.json, written by tests/golden/make_golden_dropin.py):

 * everything the reference's estimator.py imports from `network` exists on gen6d_b200.network, so the
   estimator binds this package's networks when `network` resolves to it (what a user does: put
   gen6d_b200/network on the path as `network`, or `sys.modules['network'] = gen6d_b200.network` before
   importing estimator / eval / predict);
 * every method the reference estimator calls (estimator.py:117-125,166-171,179-213) exists on our
   classes with the reference's parameter names, order and defaults;
 * `VolumeRefiner.load_ref_imgs(database, ids)` accepts a reference `BaseDatabase` as estimator.py:171
   passes it (no wrapper in user code) and the refinement host geometry runs on it.  The reference's
   `dataset.database` free functions are stood in for by the values they returned for this database."""
import inspect
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, 'golden', 'dropin_golden.json')))


def _dec(e):
    return np.asarray(e['value'], e['dtype'])


def test_reference_estimator_binds_this_package(monkeypatch):
    import gen6d_b200.network as ours
    for name in GOLD['estimator_imports']:
        assert hasattr(ours, name), name
    assert set(ours.name2network) >= {'detector', 'selector', 'refiner'}
    for name, methods in GOLD['estimator_calls'].items():
        assert set(methods) <= set(GOLD['signatures'][name]), (name, methods)

    for name, methods in GOLD['signatures'].items():
        for m, want in methods.items():
            got = inspect.signature(getattr(ours.name2network[name], m))
            w = [(p, d if has else inspect.Parameter.empty) for p, has, d in want]
            g = [(p.name, p.default) for p in got.parameters.values()]
            assert g[:len(w)] == w, (name, m, g, w)                      # same names, order, defaults ...
            assert all(d is not inspect.Parameter.empty for _, d in g[len(w):]), (name, m, g)   # ... extras are optional

    # estimator.py:171 hands the refiner a raw reference database (a CustomDatabase: no object_center attribute;
    # the reference reads centre / diameter / up vector through dataset.database's free functions)
    db = GOLD['database']
    ref_dataset = types.ModuleType('dataset')
    ref_dataset.database = types.ModuleType('dataset.database')
    ref_dataset.database.get_object_center = lambda d: _dec(db['object_center'])
    ref_dataset.database.get_diameter = lambda d: _dec(db['diameter'])[()]
    ref_dataset.database.get_object_vert = lambda d: _dec(db['object_vert'])
    monkeypatch.setitem(sys.modules, 'dataset', ref_dataset)
    monkeypatch.setitem(sys.modules, 'dataset.database', ref_dataset.database)

    from gen6d_b200.database import ReferenceDatabaseAdapter, SyntheticObjectDatabase
    from gen6d_b200 import geometry as G
    syn = SyntheticObjectDatabase(n_views=12, height=120, width=160, seed=3)

    class RefDB:            # the reference CustomDatabase's attributes and accessors (dataset/database.py:238-293)
        def __init__(self, s):
            self.database_name = 'custom/synthetic'
            self.s, self.center, self.object_point_cloud = s, s.center, s.object_point_cloud
            self.poses, self.Ks, self.img_ids = s.poses, s.Ks, s.img_ids

        def get_image(self, img_id):
            return self.s.get_image(img_id)

        def get_K(self, img_id):
            return self.Ks[img_id].copy()

        def get_pose(self, img_id):
            return self.poses[img_id].copy()

        def get_img_ids(self):
            return self.img_ids

    rdb = RefDB(syn)
    assert not hasattr(rdb, 'object_center')
    refiner = ours.name2network['refiner']({})
    refiner.load_ref_imgs(rdb, rdb.get_img_ids())                    # no adapter in user code
    assert isinstance(refiner.ref_database, ReferenceDatabaseAdapter)
    np.testing.assert_allclose(refiner.ref_database.object_center(), _dec(db['object_center']))
    assert refiner.ref_database.object_diameter() == float(_dec(db['diameter']))
    np.testing.assert_allclose(refiner.ref_database.object_vert(), _dec(db['object_vert']))
    q = rdb.get_img_ids()[5]
    a = G.refine_problem(refiner.ref_database, refiner.ref_ids, rdb.get_image(q), rdb.get_K(q), rdb.get_pose(q), 128, 6, True, warp=True)
    b = G.refine_problem(syn, syn.get_img_ids(), syn.get_image(q), syn.get_K(q), syn.get_pose(q), 128, 6, True, warp=True)
    for k in ('que_img', 'que_K', 'que_pose', 'ref_imgs', 'ref_Ks', 'ref_poses'):
        np.testing.assert_array_equal(a[k], b[k])
    # the reference's ref_info keys are a subset of ours + 'masks' (estimator.py:168; masks are unused downstream)
