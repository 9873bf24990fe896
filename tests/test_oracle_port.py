"""The NumPy port (oracle/advect_port.py) is pinned to the UNMODIFIED reference: bit-identical final
positions on every committed fixture (tests/golden/ref_*.npz, written by oracle/make_golden.py from live runs of
the reference) and on the reference's recorded results of fresh random cases."""
import numpy as np
import pytest

import common
from common import Fixture, fixtures, run_port


@pytest.mark.parametrize('name', fixtures())
def test_port_matches_reference_fixture(name):
    fx = Fixture(name)
    lon, lat, z = run_port(fx)
    assert np.array_equal(lon, fx.lon)
    assert np.array_equal(lat, fx.lat)
    assert np.array_equal(z, fx.z)
    assert np.abs(fx.lon - fx.lon0).max() > 1e-3        # the particles did move


@pytest.mark.parametrize('name', common.leeway_fixtures())
def test_leeway_port_matches_reference_fixture(name):
    fx = common.LeewayFixture(name)
    lon, lat, el = common.run_leeway_port(fx)
    assert np.array_equal(lon, fx.lon) and np.array_equal(lat, fx.lat)
    assert np.array_equal(el['orientation'], fx.orientation)
    assert np.array_equal(el['crosswind_slope'], fx.crosswind_slope)
    if fx.capsized is not None:                   # processes:capsizing: the same elements capsized
        assert np.array_equal(np.asarray(el['capsized'], dtype=np.float64), fx.capsized) and fx.capsized.sum() > 100


def test_port_matches_live_reference():
    """The port against the unmodified reference on a fresh random case (its final positions recorded in
    tests/golden/port_live_ref.npz)."""
    from oracle import advect_port as ap
    from opendrift_b200 import synthetic as syn
    g = syn.GridSpec(nx=30, ny=28, nz=6, lon0=1.0, dlon=0.07, lat0=57.0, dlat=0.04, dz=15.0)
    times = syn.slab_times(3)
    U, V = zip(*[syn.double_gyre_uv(g, (t - syn.T0).total_seconds()) for t in times])
    fields = {common.CUR[0]: np.stack(U), common.CUR[1]: np.stack(V)}
    rng = np.random.default_rng(99)
    lon = rng.uniform(1.3, 2.8, 400).astype(np.float32)
    lat = rng.uniform(57.2, 58.0, 400).astype(np.float32)
    z = rng.uniform(-80, 0, 400).astype(np.float32)

    def reference():
        from oracle import refrun
        o = refrun.run_oceandrift([refrun.make_grid_reader(g.lon, g.lat, g.z, times, fields)], lon, lat, z, syn.T0,
                                  900, 5, config={'drift:advection_scheme': 'runge-kutta4',
                                                  'drift:vertical_advection': False})
        return {'lon': o.elements.lon, 'lat': o.elements.lat}

    r = common.recorded_reference('port_live', 'rk4', reference)
    pl, pa, _ = ap.run_oceandrift([ap.GridReader(g.lon, g.lat, g.z, times, fields)], lon, lat, z, syn.T0, 900, 5)
    assert np.array_equal(pl, r['lon']) and np.array_equal(pa, r['lat'])


def _run_reference(fx):
    """The unmodified reference on a scenario object of tests/test_hostmath.py (in-memory readers of oracle/refrun.py)."""
    from oracle import refrun
    CUR = common.CUR
    m=fx.meta
    f3={CUR[0]:fx.u,CUR[1]:fx.v}
    own_w=getattr(fx,'w_lon',None) is not None
    if fx.w is not None and not own_w: f3['upward_sea_water_velocity']=fx.w
    readers=[refrun.make_grid_reader(fx.grid_lon,fx.grid_lat,fx.grid_z,fx.times,f3,'current')]
    if fx.w is not None and own_w:
        readers.append(refrun.make_grid_reader(fx.w_lon,fx.w_lat,fx.w_z,fx.times,{'upward_sea_water_velocity':fx.w},'w'))
    if fx.x_wind is not None:
        readers.append(refrun.make_grid_reader(fx.wind_lon,fx.wind_lat,None,fx.times,{'x_wind':fx.x_wind,'y_wind':fx.y_wind},'wind'))
    cfg={'drift:advection_scheme':m['scheme'],'drift:vertical_advection':bool(m['with_w']),'drift:stokes_drift':False}
    if m.get('wind_drift_depth') is not None: cfg['drift:wind_drift_depth']=m['wind_drift_depth']
    if m.get('truncate') is not None: cfg['drift:truncate_ocean_model_below_m']=m['truncate']
    if m.get('w_at_surface'): cfg['drift:vertical_advection_at_surface']=True
    kw={}
    if fx.cdf is not None: kw['current_drift_factor']=fx.cdf
    if getattr(fx,'wdf_array',None) is not None: kw['wind_drift_factor']=fx.wdf_array
    o=refrun.run_oceandrift(readers,fx.lon0,fx.lat0,fx.z0,fx.start,fx.dt,fx.steps,config=cfg,seed_kwargs=kw,seed=0)
    return o


@pytest.mark.parametrize('family,seed', [('basic', 0), ('basic', 3), ('basic', 4), ('basic', 7), ('options', 3), ('options', 6),
                                         ('options', 21), ('readers', 1), ('readers', 4), ('readers', 9), ('wdf', 1), ('wdf', 2)])
def test_port_matches_live_reference_on_random_scenarios(family, seed):
    """The port against the UNMODIFIED reference on the randomised scenarios that the device math is checked with: descending
    axes, periodic and global grids, own-grid vertical velocity, truncation, land holes, node and level particles, float32
    drift-factor arrays, backward runs.  Bit for bit, against the reference's final states recorded in
    tests/golden/port_random_ref.npz."""
    import test_hostmath as th
    fx = {'basic': th._random_scenario, 'options': th._random_options_scenario, 'readers': th._random_readers_scenario,
          'wdf': th._random_wdf_scenario}[family](seed)
    if fx is None or fx.meta.get('noise'):
        pytest.skip('scenario not applicable for this seed')

    def reference():
        o = _run_reference(fx)
        return {'lon': o.elements.lon, 'lat': o.elements.lat, 'z': o.elements.z}

    r = common.recorded_reference('port_random', '%s%d' % (family, seed), reference)
    assert len(r['lon']) == fx.n
    pl, pa, pz = common.run_port(fx)
    assert np.array_equal(pl, r['lon']) and np.array_equal(pa, r['lat'])
    assert np.array_equal(np.asarray(pz, dtype=np.float64), np.asarray(r['z'], dtype=np.float64))
