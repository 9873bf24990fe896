"""Coastline interaction (tests/coastcases.py) on the host build of the device sources: the drop-in OceanDrift with a gridded
land_binary_mask reader against runs of the unmodified reference -- surviving elements, deactivated elements in the reference's
order, their status categories ('stranded', 'seeded_on_land', 'missing_data') and positions."""
import os

import numpy as np
import pytest

import coastcases as cc
from hostengine import HostEngine


@pytest.fixture()
def host_engine(monkeypatch):
    eng = HostEngine()
    import opendrift_b200.engine as E
    import opendrift_b200.models.basemodel as B
    monkeypatch.setattr(E, 'default_engine', lambda device=None: eng)
    monkeypatch.setattr(B, 'default_engine', lambda device=None: eng)
    yield eng


@pytest.mark.parametrize('case', list(cc.CASES))
def test_coastline_case_equals_the_reference(case, host_engine):
    o = cc.run_product(case)
    n_act, n_deact, cats = cc.check(o, case)
    assert case in ('seafloor_previous', 'previous_ocean_only') or (n_deact > 0 and len(cats) > 1)
    assert 'od_coastline' in host_engine.lib.calls


def test_nearest_sampling_equals_the_reference_interpolator(host_engine):
    """od_interp + OD_INTERP_NEAREST against Nearest2DInterpolator's arithmetic (interpolators.py:26-40) restated in NumPy, float64
    and float32 positions, incl. points on and beyond the last grid point."""
    import torch
    from opendrift_b200.readers import reader_regular_grid
    from datetime import datetime
    rng = np.random.default_rng(3)
    lon, lat = np.linspace(2.0, 5.0, 23), np.linspace(58.0, 60.0, 17)
    mask = (rng.random((17, 23)) < 0.4).astype(np.float32)
    t0 = datetime(2024, 1, 1)
    r = reader_regular_grid.Reader(lon, lat, None, [t0], {'land_binary_mask': mask[None]}, name='mask')
    r.bind(host_engine)
    g, _ = r.group_of('land_binary_mask')
    n = 5000
    x = rng.uniform(2.0, 5.0, n)
    y = rng.uniform(58.0, 60.0, n)
    x[:50], y[50:100] = 5.0, 60.0
    x[100:150], y[150:200] = 2.0, 58.0
    for f32 in (False, True):
        xx = x.astype(np.float32) if f32 else x
        yy = y.astype(np.float32) if f32 else y
        got = host_engine.interp(g, t0, host_engine.to_device(xx.astype(np.float64)), host_engine.to_device(yy.astype(np.float64)),
                                 None, pos_f32=f32, raw=True, nearest=True)[0].cpu().numpy()
        xg, yg = np.asarray(r.lon_grid if hasattr(r, 'lon_grid') else lon, dtype=np.float32), np.asarray(lat, dtype=np.float32)
        xi = np.round((xx - xg.min()) / (xg.max() - xg.min()) * len(xg)).astype(np.uint32)
        yi = np.round((yy - yg.min()) / (yg.max() - yg.min()) * len(yg)).astype(np.uint32)
        xi[xi >= len(xg)] = len(xg) - 1
        yi[yi >= len(yg)] = len(yg) - 1
        cov = (xx >= xg.min()) & (xx <= xg.max()) & (yy >= yg.min()) & (yy <= yg.max())
        want = np.where(cov, mask[yi, xi], np.nan)
        assert np.array_equal(got, want, equal_nan=True)


@pytest.mark.parametrize('action,scheme,sign,out_every,release', [('stranding', 'runge-kutta4', -1, 1, 3), ('previous', 'euler', -1, 1, 0),
                                                                  ('previous', 'runge-kutta4', 1, 3, 4), ('stranding', 'runge-kutta', 1, 3, 2)])
def test_coastline_variants_against_the_live_reference(action, scheme, sign, out_every, release, host_engine):
    """Backward runs, output every third step, release over several steps: the drop-in class beside the unmodified reference's
    results on the same runs (recorded in tests/golden/coast_variants_ref.npz)."""
    from datetime import timedelta
    import common
    from opendrift_b200.models.oceandrift import OceanDrift
    from opendrift_b200.readers import reader_regular_grid

    def run(Model, make, **kw):
        fx = common.Fixture('rk4_3d')
        mlon, mlat, mask = cc.mask_grid(fx, True)
        u, v = (6 * fx.u).astype(np.float32), (6 * fx.v).astype(np.float32)
        o = Model(loglevel=50, **kw)
        o.add_reader(make(fx.grid_lon, fx.grid_lat, fx.grid_z, fx.times, {common.CUR[0]: u, common.CUR[1]: v}, 'current'))
        o.add_reader(make(mlon, mlat, None, fx.times, {'land_binary_mask': np.repeat(mask[None], len(fx.times), axis=0)}, 'mask'))
        for k, val in {'general:use_auto_landmask': False, 'environment:constant:land_binary_mask': None,
                       'general:coastline_approximation_precision': None, 'drift:vertical_advection': False, 'seed:ocean_only': False,
                       'general:coastline_action': action, 'drift:advection_scheme': scheme}.items():
            o.set_config(k, val)
        if sign > 0:
            t = fx.start if not release else [fx.start, fx.start + timedelta(seconds=release * fx.dt)]
        else:
            t = fx.times[-1] if not release else [fx.times[-1] - timedelta(seconds=release * fx.dt), fx.times[-1]]
        o.seed_elements(lon=fx.lon0[:400], lat=fx.lat0[:400], z=fx.z0[:400], time=t)
        o.run(steps=9, time_step=sign * fx.dt, time_step_output=sign * out_every * fx.dt)
        return cc.summary(o)

    def reference():
        import tempfile
        from oracle import refrun
        refrun.setup()
        from opendrift.models.oceandrift import OceanDrift as RefOD
        return run(RefOD, lambda lon, lat, z, t, f, name: refrun.make_grid_reader(lon, lat, z, t, f, name=name),
                   logfile=os.path.join(tempfile.gettempdir(), 'od_coast_live.log'))

    r = common.recorded_reference('coast_variants', '%s_%s_%d_%d_%d' % (action, scheme, sign, out_every, release), reference)
    p = run(OceanDrift, lambda lon, lat, z, t, f, name: reader_regular_grid.Reader(lon, lat, z, t, f, name=name))
    assert list(r['cats']) == list(p['cats']) and np.array_equal(r['id'], p['id'])
    assert np.array_equal(r['d_id'], p['d_id']) and np.array_equal(r['d_status'], p['d_status']) and len(r['d_id']) > 0
    assert max(common.max_err_deg(p['lon'], p['lat'], r['lon'], r['lat'])) < 5e-8
    assert max(common.max_err_deg(p['d_lon'], p['d_lat'], r['d_lon'], r['d_lat'])) < 5e-8
