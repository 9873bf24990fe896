"""BASELINE configs[0] on the CPU: the reference's analytical double-gyre reader on its stereographic plane
(examples/example_double_gyre_advection_schemes.py).

  * the oracle pieces that stand in for pyproj (oracle/proj_stere.py, Geod.inv of oracle/geod_karney.py) against mpmath;
  * the NumPy port (oracle/gyre_port.py + oracle/advect_port.py) against the fixtures the UNMODIFIED reference produced
    (tests/golden/ref_gyre_*.npz, oracle/make_golden.py), bit for bit, and against its recorded runs on random cases;
  * the device code (opendrift_b200/csrc/od_analytic.cuh) compiled for the host against the oracle and the fixtures.

Tolerance.  The box is 2 m x 1 m at (0 E, 0 N): 1e-6 deg (the north-star tolerance) is 0.11 m there, 5 % of the domain,
so these tests hold 1e-9 deg (1.1e-4 m).  Measured: <= 1.2e-5 m after 60 RK4 steps -- sampling is bit-identical
(test_sampler_matches_port); what remains is the ~1e-9 m at which any two implementations of the geodesic agree per
move (and NumPy's float32 arctan2), amplified by the gyre's chaotic stretching."""
import ctypes as C
import os
from datetime import timedelta

import numpy as np
import pytest

import common
import gyre_common as gc
from opendrift_b200 import _lib

TOL_M = 1.1e-4          # 1e-9 deg on the ground


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


# ---- the oracle's stand-ins for pyproj -------------------------------------------------------------------------
@pytest.mark.parametrize('proj4', [
    '+proj=stere +lat_0=0 +lon_0=0 +lat_ts=0 +units=m +a=6.371e+06 +e=0 +no_defs',
    '+proj=stere +lat_0=60 +lon_0=10 +R=6371000 +x_0=1000 +y_0=-2000 +units=m +no_defs',
    '+proj=stere +lat_0=90 +lon_0=70 +lat_ts=60 +R=6371000 +units=m +no_defs',
    '+proj=stere +lat_0=-90 +lon_0=0 +R=6371000 +units=m +no_defs'])
def test_stereographic_oracle_against_mpmath(proj4):
    """Closed form (Snyder 21-2..21-4: x = R k cos(phi) sin(dlam), y = R k [cos(phi1) sin(phi) - sin(phi1) cos(phi) cos(dlam)],
    k = 2 k0 / (1 + sin(phi1) sin(phi) + cos(phi1) cos(phi) cos(dlam))) at 40 digits; polar scale for lat_ts from 21-7/21-11."""
    import mpmath as mp
    from oracle.proj_stere import Stere, parse_proj4
    mp.mp.dps = 40
    P = Stere(proj4)
    p = parse_proj4(proj4)
    R = mp.mpf(p.get('R', p.get('a')))
    phi1, lam0 = mp.radians(mp.mpf(p['lat_0'])), mp.radians(mp.mpf(p['lon_0']))
    k0 = mp.mpf(1)
    if abs(p['lat_0']) == 90 and 'lat_ts' in p:                   # true scale at lat_ts: k0 = (1 + sin|lat_ts|) / 2
        k0 = (1 + mp.sin(mp.radians(abs(mp.mpf(p['lat_ts']))))) / 2
    rng = np.random.default_rng(3)
    lon = p['lon_0'] + rng.uniform(-40, 40, 60)
    lat = np.clip(p['lat_0'] + rng.uniform(-35, 35, 60), -89.5, 89.5)
    x, y = P.forward(lon, lat)
    for i in range(len(lon)):
        phi, dl = mp.radians(mp.mpf(float(lat[i]))), mp.radians(mp.mpf(float(lon[i]))) - lam0
        k = 2 * k0 / (1 + mp.sin(phi1) * mp.sin(phi) + mp.cos(phi1) * mp.cos(phi) * mp.cos(dl))
        ex = R * k * mp.cos(phi) * mp.sin(dl) + mp.mpf(p.get('x_0', 0.0))
        ey = R * k * (mp.cos(phi1) * mp.sin(phi) - mp.sin(phi1) * mp.cos(phi) * mp.cos(dl)) + mp.mpf(p.get('y_0', 0.0))
        assert abs(float(ex) - x[i]) < 2e-8 and abs(float(ey) - y[i]) < 2e-8, (i, float(ex), x[i], float(ey), y[i])
    lo, la = P.inverse(x, y)                                       # round trip
    assert np.max(np.abs((lo - lon + 180) % 360 - 180)) < 1e-12 and np.max(np.abs(la - lat)) < 1e-12


def test_gyre_seed_point_of_the_example():
    """examples/example_double_gyre_advection_schemes.py: xy2lonlat(0.6, 0.3) on the reader's plane; at the origin of
    an equatorial stereographic projection lon = x / R and lat = y / R to 1e-14 relative."""
    from oracle.proj_stere import Stere
    P = Stere('+proj=stere +lat_0=0 +lon_0=0 +lat_ts=0 +units=m +a=6.371e+06 +e=0 +no_defs')
    lon, lat = P.inverse(np.array([0.6]), np.array([0.3]))
    assert lon[0] == pytest.approx(np.degrees(0.6 / 6.371e6), rel=1e-12)
    assert lat[0] == pytest.approx(np.degrees(0.3 / 6.371e6), rel=1e-12)
    fx = gc.GyreFixture('gyre_example_rk4_dt01')                  # what the reference run was seeded with
    assert fx.seed_lon[0] == lon[0] and fx.seed_lat[0] == lat[0]


def test_inverse_geodesic_oracle_against_exact_integrals():
    """Geod.inv stand-in (oracle/geod_karney.py:inverse_short): end points from the series-free mpmath solution of the
    direct problem (oracle/geod_exact.py); the recovered azimuth and distance must reproduce the line."""
    from oracle import geod_karney as gk
    from oracle.geod_exact import direct_exact
    rng = np.random.default_rng(11)
    n = 24
    lon1, lat1 = rng.uniform(-180, 180, n), rng.uniform(-80, 80, n)
    az, s = rng.uniform(-180, 180, n), np.concatenate([np.full(8, 10.0), rng.uniform(1, 5e4, n - 8)])
    end = np.array([direct_exact(*c) for c in zip(lon1, lat1, az, s)])
    a1, _, ss = gk.inverse_short(lon1, lat1, end[:, 0], end[:, 1])
    d = np.radians((a1 - az + 180) % 360 - 180)
    assert np.max(np.abs(d * s)) < 2e-8          # cross-track miss in metres (end-point coordinates carry ~3e-9 m of round-off)
    assert np.max(np.abs(ss - s)) < 2e-8
    f, b, dist = gk.Geod().inv(4.0, 60.0, 4.0, 60.1)
    assert abs(f) < 1e-9 and abs(abs(b) - 180) < 1e-9 and dist == pytest.approx(11141.5, abs=1.0)


# ---- the port against the reference --------------------------------------------------------------------------------
@pytest.mark.parametrize('name', gc.gyre_fixtures())
def test_port_matches_reference_fixture_bit_for_bit(name):
    fx = gc.GyreFixture(name)
    lon, lat = gc.run_port(fx)
    assert np.array_equal(lon, fx.lon) and np.array_equal(lat, fx.lat)


def test_port_matches_live_reference_random_gyre():
    """The port against the unmodified reference's double-gyre runs on random parameters and seeds (recorded in
    tests/golden/gyre_random_ref.npz: the seeds the reference's reader placed and its final positions)."""
    from datetime import datetime
    from oracle import advect_port as ap, gyre_port
    rng = np.random.default_rng(5)
    for scheme, dt, n in (('runge-kutta4', 0.07, 300), ('runge-kutta', -0.05, 200), ('euler', 0.2, 1)):
        eps, om, A = rng.uniform(0.05, 0.3), rng.uniform(0.3, 1.0), rng.uniform(0.1, 0.3)
        x, y = rng.uniform(-0.02, 2.02, n), rng.uniform(-0.02, 1.02, n)

        def reference():
            import tempfile
            from oracle import refrun
            refrun.setup()
            from opendrift.readers import reader_double_gyre
            from opendrift.models.oceandrift import OceanDrift
            dg = reader_double_gyre.Reader(epsilon=eps, omega=om, A=A)
            lon, lat = dg.xy2lonlat(x, y)
            o = OceanDrift(loglevel=50, logfile=os.path.join(tempfile.gettempdir(), 'od_gyre_test.log'))
            o.set_config('environment:fallback:land_binary_mask', 0)
            o.set_config('general:use_auto_landmask', False)
            o.set_config('drift:advection_scheme', scheme)
            o.add_reader(dg)
            o.seed_elements(lon, lat, time=dg.initial_time)
            o.run(steps=25, time_step=dt)
            return {'seed_lon': lon, 'seed_lat': lat, 'initial_time': dg.initial_time.isoformat(), 'steps': o.steps_calculation,
                    'lon': o.elements.lon, 'lat': o.elements.lat}

        r = common.recorded_reference('gyre_random', scheme, reference)
        t0 = datetime.fromisoformat(str(r['initial_time']))
        pr = gyre_port.DoubleGyreReader(t0, epsilon=eps, omega=om, A=A)
        # (the reference runs int(duration / time_step) steps: 24 for 25 * 0.07 s)
        pl, pa, _ = ap.run_oceandrift([pr], r['seed_lon'], r['seed_lat'], np.zeros(n), t0, dt, int(r['steps']), scheme=scheme)
        assert np.array_equal(pl, r['lon']) and np.array_equal(pa, r['lat']), scheme


# ---- the device code, compiled for the host ----------------------------------------------------------------------------
def _desc(fx, fallback=False):
    rd = fx.product_reader()
    if fallback:
        rd.bind(None, {v: 0.0 for v in rd.variables})
    return rd, rd.analytic_desc(with_fallback=fallback)


def test_device_projection_and_azimuth_match_oracle():
    lib = common.hostshim()
    fx = gc.GyreFixture('gyre_rk4')
    rd, d = _desc(fx)
    pr = fx.port_reader()
    rng = np.random.default_rng(2)
    n = 20000
    x, y = rng.uniform(-5, 5, n), rng.uniform(-5, 5, n)
    lon, lat = pr.proj.inverse(x, y)
    hl, ha, hx, hy = (np.empty(n) for _ in range(4))
    lib.hs_stere(C.byref(d), 1, C.c_int64(n), _vp(x), _vp(y), _vp(hl), _vp(ha))
    assert np.max(np.abs(hl - lon)) < 1e-20 and np.max(np.abs(ha - lat)) < 1e-20         # degrees; values ~1e-5
    lib.hs_stere(C.byref(d), 0, C.c_int64(n), _vp(lon), _vp(lat), _vp(hx), _vp(hy))
    ox, oy = pr.proj.forward(lon, lat)
    assert np.max(np.abs(hx - ox)) < 1e-14 and np.max(np.abs(hy - oy)) < 1e-14           # metres
    # the product's host-side projection (seeding helper) agrees with both
    px, py = rd.lonlat2xy(lon, lat)
    assert np.max(np.abs(px - ox)) < 1e-14 and np.max(np.abs(py - oy)) < 1e-14
    # forward azimuth of short lines anywhere on the ellipsoid
    from oracle import geod_karney as gk
    lon1, lat1 = rng.uniform(-180, 180, n), rng.uniform(-85, 85, n)
    az, s = rng.uniform(-180, 180, n), rng.uniform(1.0, 100.0, n)          # rotate_vectors uses a 10 m line
    lon2, lat2 = gk.direct(lon1, lat1, az, s)
    oaz = np.radians(gk.inverse_short(lon1, lat1, lon2, lat2)[0])
    haz = np.empty(n)
    lib.hs_inverse_azimuth(C.c_int64(n), _vp(lon1), _vp(lat1), _vp(lon2), _vp(lat2), _vp(haz))
    d_az = (haz - oaz + np.pi) % (2 * np.pi) - np.pi
    assert np.max(np.abs(d_az * s)) < 1e-8        # metres across the line: the round-off of the end-point coordinates


def test_sampler_matches_port():
    """Reader chain for one get_environment call: float32 velocities bit for bit, NaN mask identical."""
    lib = common.hostshim()
    fx = gc.GyreFixture('gyre_rk4')
    rd, d = _desc(fx)
    pr = fx.port_reader()
    rng = np.random.default_rng(0)
    n = 50000
    lon, lat = rd.xy2lonlat(rng.uniform(-0.02, 2.02, n), rng.uniform(-0.02, 1.02, n))
    for tsec, f32 in ((0.0, False), (1.35, False), (4.2, True)):
        lo = lon.astype(np.float32) if f32 else lon
        la = lat.astype(np.float32) if f32 else lat
        e = pr.interpolate(common.CUR, fx.t0 + timedelta(seconds=tsec), lo, la, None)
        pu, pv = (e[k].astype(np.float32) for k in common.CUR)
        u, v = np.empty(n, np.float32), np.empty(n, np.float32)
        lo64, la64 = lo.astype(np.float64), la.astype(np.float64)
        assert lib.hs_analytic_interp(C.byref(d), C.c_double(tsec), C.c_int64(n), _vp(lo64), _vp(la64), 1 if f32 else 0,
                                      _vp(u), _vp(v)) == 0
        assert np.array_equal(np.isnan(u), np.isnan(pu)) and 0 < np.isnan(u).sum() < n / 10
        ok = ~np.isnan(u)
        ulp = np.spacing(np.abs(pu[ok]).max())
        assert np.max(np.abs(u[ok] - pu[ok])) <= ulp and np.max(np.abs(v[ok] - pv[ok])) <= ulp
        assert np.mean(u[ok] == pu[ok]) > 0.999 and np.mean(v[ok] == pv[ok]) > 0.999


@pytest.mark.parametrize('mode', [_lib.OD_MATH_SERIES, _lib.OD_MATH_EXACT, _lib.OD_MATH_FAST])
@pytest.mark.parametrize('name', gc.gyre_fixtures())
def test_device_math_matches_reference_fixture(name, mode):
    fx = gc.GyreFixture(name)
    lon, lat = gc.run_hostshim(fx, mode)
    err = gc.plane_error_m(fx, lon, lat, fx.lon, fx.lat)
    assert err < TOL_M, err


def test_descriptor_errors():
    lib = common.hostshim()
    fx = gc.GyreFixture('gyre_rk4')
    rd, d = _desc(fx)
    z = np.zeros(1)
    o = np.zeros(1, np.float32)
    d.kind = 7
    assert lib.hs_analytic_interp(C.byref(d), C.c_double(0), C.c_int64(1), _vp(z), _vp(z), 0, _vp(o), _vp(o)) == -1
    d = rd.analytic_desc()
    d.proj.kind = 9
    assert lib.hs_analytic_interp(C.byref(d), C.c_double(0), C.c_int64(1), _vp(z), _vp(z), 0, _vp(o), _vp(o)) == -2
    d = rd.analytic_desc()
    d.proj.a = 0.0
    assert lib.hs_analytic_interp(C.byref(d), C.c_double(0), C.c_int64(1), _vp(z), _vp(z), 0, _vp(o), _vp(o)) == -3
    from opendrift_b200.readers.reader_double_gyre import Reader
    with pytest.raises(NotImplementedError):
        Reader(proj4='+proj=stere +lat_0=90 +lon_0=0 +ellps=WGS84')           # ellipsoidal: not on the GPU path
    with pytest.raises(NotImplementedError):
        Reader(proj4='+proj=lcc +lat_1=60 +lat_2=65 +R=6371000')


# ---- the drop-in classes on the host build (tests/hostengine.py): model glue, reader glue, Engine's argument structs ----
def _model(fx, eng, arithmetic=None):
    from opendrift_b200.models.oceandrift import OceanDrift
    o = OceanDrift(loglevel=50, engine=eng)
    o.set_config('environment:fallback:land_binary_mask', 0)
    o.set_config('general:use_auto_landmask', False)
    o.set_config('drift:advection_scheme', fx.scheme)
    if arithmetic:
        o.set_config('gpu:arithmetic', arithmetic)
    rd = fx.product_reader()
    o.add_reader(rd)
    kw = {} if fx.cdf is None else {'current_drift_factor': fx.cdf}
    o.seed_elements(fx.seed_lon, fx.seed_lat, time=rd.initial_time, **kw)
    return o, rd


@pytest.mark.parametrize('name', gc.gyre_fixtures())
def test_dropin_model_runs_the_example(name):
    """OceanDrift + reader_double_gyre.Reader exactly as examples/example_double_gyre_advection_schemes.py uses them
    (add_reader, seed_elements, run), with the engine swapped for the host build of the device code."""
    from hostengine import HostEngine
    fx = gc.GyreFixture(name)
    eng = HostEngine()
    o, rd = _model(fx, eng)
    o.run(steps=fx.steps, time_step=fx.dt)
    lon, lat = np.asarray(o.elements.lon), np.asarray(o.elements.lat)
    assert o.steps_calculation == fx.steps and lon.dtype == np.float64
    assert gc.plane_error_m(fx, lon, lat, fx.lon, fx.lat) < TOL_M
    hl, ha = gc.run_hostshim(fx)                      # the same steps through the C-ABI structs directly
    assert np.array_equal(lon, hl) and np.array_equal(lat, ha)
    assert eng.lib.calls.count('od_analytic_advect') == fx.steps        # one launch per step for the stage loop
    x, y = rd.lonlat2xy(lon, lat)                     # the script's way of reading results back
    assert np.all(np.isfinite(x)) and x.min() > -0.1 and x.max() < 2.1 and y.min() > -0.1 and y.max() < 1.1


def test_dropin_duration_and_arithmetic_modes():
    from hostengine import HostEngine
    from datetime import timedelta as td
    fx = gc.GyreFixture('gyre_example_rk4_dt01')
    res = {}
    for mode in ('series', 'exact', 'fast'):
        o, _ = _model(fx, HostEngine(), arithmetic=mode)
        o.run(duration=td(seconds=6), time_step=0.1)             # the example's call
        assert o.steps_calculation == 60
        res[mode] = (np.asarray(o.elements.lon), np.asarray(o.elements.lat))
        assert gc.plane_error_m(fx, res[mode][0], res[mode][1], fx.lon, fx.lat) < TOL_M
    assert not np.array_equal(res['series'][0], res['exact'][0])    # the modes really are different code paths


def test_reader_and_environment_calls_on_host_engine():
    """Reader.get_variables_interpolated and Environment.get_environment (the reference's signatures) for the
    analytical reader: float32 values of the port, masked / fallback where uncovered."""
    from hostengine import HostEngine
    fx = gc.GyreFixture('gyre_rk4')
    eng = HostEngine()
    o, rd = _model(fx, eng)
    pr = fx.port_reader()
    t = fx.t0 + timedelta(seconds=2.5)
    rng = np.random.default_rng(8)
    lon, lat = rd.xy2lonlat(rng.uniform(-0.05, 2.05, 4000), rng.uniform(-0.05, 1.05, 4000))
    rd.bind(eng)
    env, prof = rd.get_variables_interpolated(common.CUR, time=t, lon=lon, lat=lat, z=0, rotate_to_proj='+proj=latlong')
    e = pr.interpolate(common.CUR, t, lon, lat, None)
    for k in common.CUR:
        ref = e[k].astype(np.float32)
        assert np.array_equal(np.ma.getmaskarray(env[k]), np.isnan(ref)) and np.isnan(ref).sum() > 50
        ok = ~np.isnan(ref)
        assert np.array_equal(np.asarray(env[k])[ok], ref[ok])
    assert prof is None
    from opendrift_b200.errors import OutsideSpatialCoverageError
    with pytest.raises(OutsideSpatialCoverageError):
        rd.get_variables_interpolated(common.CUR, time=t, lon=np.array([10.0]), lat=np.array([10.0]))
    # Environment.get_environment: fallback 0 where the reader does not cover
    o.env.finalize(eng)
    renv, _, missing = o.env.get_environment(common.CUR, t, lon, lat, np.zeros(len(lon)))
    for k in common.CUR:
        ref = e[k].astype(np.float32)
        ref[np.isnan(ref)] = 0.0
        assert np.array_equal(renv[k], ref)
    assert not missing.any()


# ---- the other aspects of the projection (oblique, north / south polar) in a whole run -----------------------------------
@pytest.mark.parametrize('proj4', gc.ASPECTS)
def test_other_projection_aspects_whole_run(proj4):
    """The double gyre placed on oblique and polar stereographic planes and across the dateline: host-compiled device
    code against the port, and the port against the unmodified reference's results (tests/golden/gyre_aspects_ref.npz).
    (At these latitudes the float32 seed arrays of the reference quantise the 2 m box to a few distinct positions -- parity
    is what is checked, not oceanography.  Readers north of 89 deg are discarded by the reference's simulation extent,
    basemodel/__init__.py:2026-2034, hence the offsets.)"""
    fx = gc.AspectCase(proj4)
    sx, sy = fx.plane.forward(fx.seed_lon.astype(np.float32).astype(np.float64), fx.seed_lat.astype(np.float32).astype(np.float64))
    px, py = fx.plane.forward(fx.lon, fx.lat)
    assert np.hypot(px - sx, py - sy).max() > 0.3                # the particles really travelled
    hl, ha = gc.run_hostshim(fx)
    assert fx.error_m(hl, ha) < 1e-5
    from hostengine import HostEngine
    o, _ = _model(fx, HostEngine())                              # the drop-in classes on the host build
    o.run(steps=fx.steps, time_step=fx.dt)
    assert np.array_equal(np.asarray(o.elements.lon), hl) and np.array_equal(np.asarray(o.elements.lat), ha)

    def reference():
        import tempfile
        from oracle import refrun
        refrun.setup()
        from opendrift.readers import reader_double_gyre
        from opendrift.models.oceandrift import OceanDrift
        dg = reader_double_gyre.Reader(initial_time=fx.t0, proj4=proj4, **fx.par)
        o = OceanDrift(loglevel=50, logfile=os.path.join(tempfile.gettempdir(), 'od_gyre_test.log'))
        o.set_config('environment:fallback:land_binary_mask', 0)
        o.set_config('general:use_auto_landmask', False)
        o.set_config('drift:advection_scheme', fx.scheme)
        o.add_reader(dg)
        o.seed_elements(fx.seed_lon, fx.seed_lat, time=fx.t0)
        o.run(steps=fx.steps, time_step=fx.dt)
        return {'steps': o.steps_calculation, 'lon': o.elements.lon, 'lat': o.elements.lat}

    r = common.recorded_reference('gyre_aspects', 'aspect%d' % gc.ASPECTS.index(proj4), reference)
    assert int(r['steps']) == fx.steps
    assert np.array_equal(fx.lon, r['lon']) and np.array_equal(fx.lat, r['lat'])


def test_bench_extra_measurement_runs_on_host_engine():
    """bench.py's guarded configs[0] measurement (timing aside): same code with the host engine and a stub for the CUDA events."""
    import time
    import types
    import bench
    from hostengine import HostEngine

    class Ev:
        def __init__(self, enable_timing=True):
            self.t = 0.0

        def record(self):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3
    fake = types.SimpleNamespace(cuda=types.SimpleNamespace(Event=Ev, synchronize=lambda: None))
    r = bench.configs0_double_gyre(HostEngine(), fake, 20000)
    assert r['parity_ok'] and r['max_err_m_vs_port_one_step'] < 1e-7
    assert r['kernel_ms'] > 0 and r['algorithmic_bytes_per_launch'] == 32 * 20000 and r['cpu_port_particle_steps_per_s'] > 0
