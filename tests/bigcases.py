"""The BENCHMARKED configurations (BASELINE.json configs[1], [3], [4]: the 512 x 512 x 50 u/v/w reader with RK4; the 3-D current +
wind + Stokes + vertical-mixing set; Leeway / Euler) at 1e5 particles, against results of the UNMODIFIED reference
(tests/golden/ref_big_*.npz, written by `python -m oracle.make_golden big`).  The forcing is regenerated from
opendrift_b200/synthetic.py -- the same formulas the generator handed to the reference; the fixtures hold the configuration and the
reference's final state of a fixed sample of the elements only (oracle/make_golden.py:big_sample_ids)."""
import json
import os
from datetime import timedelta

import numpy as np

import common
from oracle.make_golden import BIG, BIG_N, big_fields       # (pure NumPy; the reference is only touched by run_big_case)
from opendrift_b200 import synthetic as syn

KINDS = [k for k in BIG if os.path.exists(os.path.join(common.GOLDEN, 'ref_big_%s.npz' % k))]


class BigCase:
    def __init__(self, kind):
        d = np.load(os.path.join(common.GOLDEN, 'ref_big_%s.npz' % kind))
        self.kind, self.meta = kind, json.loads(str(d['meta']))
        self.ref = {k: d[k] for k in d.files if k != 'meta'}
        c = self.meta
        assert c['n'] == BIG_N and c['steps'] == BIG[kind]['steps'] and c['config'] == BIG[kind]['config'], 'fixture is stale'
        self.grid, self.times, self.fields = big_fields(kind, c['n_slabs'])
        self.lon0, self.lat0, self.z0 = syn.particle_cloud(BIG_N, seed=c['seed'], three_d=self.grid.z is not None)
        self.start = syn.T0 + timedelta(seconds=c['start_offset_s'])
        self.steps, self.dt = c['steps'], c['dt']

    def model(self, subset=None, **cfg):
        """The drop-in model class, readers added, configured and seeded as the generator drove the reference."""
        from opendrift_b200.readers import reader_regular_grid
        c, g = self.meta, self.grid
        if c['model'] == 'Leeway':
            from opendrift_b200.models.leeway import Leeway as Model
        else:
            from opendrift_b200.models.oceandrift import OceanDrift as Model
        o = Model(loglevel=50, seed=0)
        for nm, f in self.fields.items():
            o.add_reader(reader_regular_grid.Reader(g.lon, g.lat, g.z if nm == 'current' else None, self.times, f, name=nm))
        o.set_config('general:use_auto_landmask', False)
        o.set_config('general:coastline_action', 'none')
        for k, v in c['config'].items():
            o.set_config(k, v)
        for k, v in cfg.items():
            o.set_config(k, v)
        s = slice(None) if subset is None else subset
        if c['model'] == 'Leeway':
            o.seed_elements(lon=self.lon0[s], lat=self.lat0[s], time=self.start, object_type=c['object_type'])
        else:
            o.seed_elements(lon=self.lon0[s], lat=self.lat0[s], z=self.z0[s], time=self.start)
        return o

    def check(self, o, tol_deg=5e-8, z_tol=0.0):
        """A run of all BIG_N elements against the reference's final state of the stored sample."""
        ref, s = self.ref, self.ref['ids']
        assert o.num_elements_active() == self.meta['n']
        ids = np.asarray(o.elements.ID)
        assert np.array_equal(ids, np.arange(len(ids)))
        e = common.max_err_deg(np.asarray(o.elements.lon)[s], np.asarray(o.elements.lat)[s], ref['lon'], ref['lat'])
        assert max(e) < tol_deg, e
        out = {'max_err_deg': max(e)}
        if 'z' in ref:
            z = np.asarray(o.elements.z)[s]
            assert z.dtype == ref['z'].dtype
            dz = float(np.abs(z.astype(np.float64) - ref['z'].astype(np.float64)).max())
            assert dz <= z_tol, dz
            out['max_err_z'] = dz
        if 'orientation' in ref:
            assert np.array_equal(np.asarray(o.elements.orientation).astype(np.int8)[s], ref['orientation'])
        return out
