"""Ensemble blocks (tests/enscases.py) on the host build of the device sources: the drop-in OceanDrift against runs of the unmodified
reference on the same ensemble reader -- member i % n_members per element, also when a second reader serves part of the elements;
and the reference's own known answer for ReaderBlock with ensemble members (tests/readers/test_interpolation.py:231-259)."""
import os

import numpy as np
import pytest

import enscases as ec
from hostengine import HostEngine


@pytest.fixture()
def host_engine(monkeypatch):
    eng = HostEngine()
    import opendrift_b200.engine as E
    import opendrift_b200.models.basemodel as B
    monkeypatch.setattr(E, 'default_engine', lambda device=None: eng)
    monkeypatch.setattr(B, 'default_engine', lambda device=None: eng)
    yield eng


@pytest.mark.parametrize('case', list(ec.CASES))
def test_ensemble_case_equals_the_reference(case, host_engine):
    o = ec.run_product(case)
    e, spread = ec.check(o, case)
    assert e < 5e-8, e
    assert spread > 100 * 5e-8          # the members differ by far more than the tolerance


def test_reference_known_answer_for_ensemble_members(host_engine):
    """test_interpolation_ensemble: members 1, 2, 3 (2-D) and 31, 32, 33 (3-D): element 0 -> member 0, 1 -> 1, 3 -> 0."""
    from datetime import datetime
    lon, lat, z = np.linspace(2, 6, 20), np.linspace(58, 61, 16), np.array([0.0, -10.0, -30.0])
    t0 = datetime(2024, 1, 1)
    one2, one3 = np.ones((1, 16, 20), dtype=np.float32), np.ones((1, 3, 16, 20), dtype=np.float32)
    r2 = ec.product_ensemble_reader(lon, lat, None, [t0], {'x_wind': [one2 * 1, one2 * 2, one2 * 3]}, 'e2')
    r3 = ec.product_ensemble_reader(lon, lat, z, [t0], {'sea_water_temperature': [one3 * 31, one3 * 32, one3 * 33]}, 'e3')
    r2.bind(host_engine)
    r3.bind(host_engine)
    x, y, zz = np.linspace(2.5, 5.5, 15), np.linspace(58.5, 60.5, 15), -np.linspace(0, 25, 15)
    v2 = r2.get_variables_interpolated(['x_wind'], time=t0, lon=x, lat=y, z=zz)[0]['x_wind']
    v3 = r3.get_variables_interpolated(['sea_water_temperature'], time=t0, lon=x, lat=y, z=zz)[0]['sea_water_temperature']
    assert (v2[0], v2[1], v2[3]) == (1, 2, 1)
    assert v3[0] == 31 and v3[1] == 32 and abs(v3[3] - 31) < 1e-12
    assert list(v2) == [1 + (i % 3) for i in range(15)]


@pytest.mark.parametrize('n_ens,scheme,release,max_age,wind_ens', [(2, 'runge-kutta4', 4, 0, False), (5, 'runge-kutta', 0, 0, True),
                                                                   (2, 'runge-kutta4', 5, 2500, True)])
def test_ensemble_variants_against_the_live_reference(n_ens, scheme, release, max_age, wind_ens, host_engine):
    """Release over several steps and retirement change an element's rank among the served positions from step to step; a wind
    reader with its own number of members: the drop-in class beside the unmodified reference's results on the same runs (recorded in
    tests/golden/ensemble_variants_ref.npz)."""
    from datetime import timedelta
    import common
    from opendrift_b200.models.oceandrift import OceanDrift

    def run(Model, mk_ens, **kw):
        fx = common.Fixture('rk4_3d')
        us = [((1 + 0.5 * m) * fx.u).astype(np.float32) for m in range(n_ens)]
        vs = [((1 - 0.3 * m) * fx.v).astype(np.float32) for m in range(n_ens)]
        o = Model(loglevel=50, **kw)
        o.add_reader(mk_ens(fx.grid_lon, fx.grid_lat, fx.grid_z, fx.times, {common.CUR[0]: us, common.CUR[1]: vs}, 'ens'))
        if wind_ens:
            nt, ny, nx = len(fx.times), len(fx.grid_lat), len(fx.grid_lon)
            X, Y = np.meshgrid(np.linspace(0, 1, nx), np.linspace(0, 1, ny))
            wx = [np.stack([(6 + 3 * m) * np.cos(0.3 * k) * (1 + 0.2 * X) for k in range(nt)]).astype(np.float32) for m in range(4)]
            wy = [np.stack([(6 + 3 * m) * np.sin(0.3 * k) * (1 + 0.2 * Y) for k in range(nt)]).astype(np.float32) for m in range(4)]
            o.add_reader(mk_ens(fx.grid_lon, fx.grid_lat, None, fx.times, {'x_wind': wx, 'y_wind': wy}, 'wens'))
        cfg = {'general:use_auto_landmask': False, 'general:coastline_action': 'none', 'drift:vertical_advection': False,
               'drift:advection_scheme': scheme}
        if max_age:
            cfg['drift:max_age_seconds'] = max_age
        for k, v in cfg.items():
            o.set_config(k, v)
        if 'environment:constant:land_binary_mask' in getattr(o, '_config', {}):
            o.set_config('environment:constant:land_binary_mask', 0)
        t = fx.start if not release else [fx.start, fx.start + timedelta(seconds=release * fx.dt)]
        o.seed_elements(lon=fx.lon0[:401], lat=fx.lat0[:401], z=np.where(np.arange(401) % 2 == 0, 0.0, fx.z0[:401]), time=t, wind_drift_factor=0.03)
        o.run(steps=8, time_step=fx.dt, time_step_output=fx.dt)
        return np.asarray(o.elements.ID), np.asarray(o.elements.lon, dtype=np.float64), np.asarray(o.elements.lat, dtype=np.float64)

    def reference():
        import tempfile
        from oracle import refrun
        refrun.setup()
        from opendrift.models.oceandrift import OceanDrift as RefOD
        return dict(zip(('id', 'lon', 'lat'), run(RefOD, ec.reference_ensemble_reader,
                                                  logfile=os.path.join(tempfile.gettempdir(), 'ens_live.log'))))

    rec = common.recorded_reference('ensemble_variants', '%d_%s_%d_%d_%d' % (n_ens, scheme, release, max_age, wind_ens), reference)
    r = rec['id'], rec['lon'], rec['lat']
    p = run(OceanDrift, ec.product_ensemble_reader)
    assert np.array_equal(r[0], p[0]) and len(r[0]) > 0
    assert max(common.max_err_deg(p[1], p[2], r[1], r[2])) < 5e-8
