"""ORACLE fixture generator: runs the UNMODIFIED reference (oracle/refrun.py, this container
only) on small seeded cases and writes inputs + final positions to tests/golden/ref_*.npz.

    python -m oracle.make_golden

The fixtures travel to the GPU box; /root/reference does not.  Each fixture stores the
complete forcing (float32 slabs), the seeded particles, the configuration and the
reference's final lon/lat/z (float64/float64/float32).
"""
import json
from datetime import timedelta
import os

import numpy as np

from oracle import refrun
from opendrift_b200 import synthetic as syn

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'tests', 'golden')

CURRENT = ['x_sea_water_velocity', 'y_sea_water_velocity']


def build_fields(g, n_slabs, with_w=False, mixing=False):
    times = syn.slab_times(n_slabs)
    U, V = [], []
    for t in times:
        u, v = syn.double_gyre_uv(g, (t - syn.T0).total_seconds(), three_d=g.z is not None)
        U.append(u)
        V.append(v)
    f = {CURRENT[0]: np.stack(U), CURRENT[1]: np.stack(V)}
    if with_w:
        f['upward_sea_water_velocity'] = np.stack([syn.upward_w(g)] * n_slabs)
    if mixing:
        f['ocean_vertical_diffusivity'] = np.stack([syn.vertical_diffusivity(g, (t - syn.T0).total_seconds()) for t in times])
    return times, f


def punch_holes(g, fields):
    """Land: an island (NaN in every layer), a 'coast' band and a shoaling sea floor (NaN in the deep layers)."""
    iy, ix = np.meshgrid(np.arange(g.ny), np.arange(g.nx), indexing='ij')
    island = (ix - 20) ** 2 + (iy - 18) ** 2 <= 10
    coast = ix >= g.nx - 4
    shoal = (ix - 9) ** 2 + (iy - 9) ** 2 <= 30
    for k in (CURRENT[0], CURRENT[1]):
        a = fields[k]
        if a.ndim == 4:
            a[:, :, island | coast] = np.nan
            a[:, a.shape[1] - 3:, shoal] = np.nan
        else:
            a[:, island | coast] = np.nan


def build_stokes(g, n_slabs, with_hs):
    times = syn.slab_times(n_slabs)
    sx, sy = zip(*[syn.stokes_xy(g, (t - syn.T0).total_seconds()) for t in times])
    f = {'sea_surface_wave_stokes_drift_x_velocity': np.stack(sx), 'sea_surface_wave_stokes_drift_y_velocity': np.stack(sy)}
    if with_hs:
        f['sea_surface_wave_significant_height'] = np.stack([syn.wave_height(g, 0.0)] * n_slabs)
    return f


def build_wind(g, n_slabs):
    times = syn.slab_times(n_slabs)
    X, Y = [], []
    for t in times:
        wx, wy = syn.wind_xy(g, (t - syn.T0).total_seconds())
        X.append(wx)
        Y.append(wy)
    return {'x_wind': np.stack(X), 'y_wind': np.stack(Y)}


def run_case(name, g, n, steps, dt, scheme, with_w=False, wind=False, diffusivity=0.0,
             cdf=None, spill=False, seed=0, wind_drift_depth=None, start_offset_s=0, mixing=False, dt_mix=60.0, stokes=None, stokes_hs=True, holes=False, noise=None,
             truncate=None, w_at_surface=False, diffusivity_model=None, background_diffusivity=None):
    n_slabs = syn.n_slabs_for(steps, dt) + (1 if start_offset_s else 0)
    times, f3 = build_fields(g, n_slabs, with_w, mixing and diffusivity_model in (None, 'environment'))
    if holes:
        punch_holes(g, f3)
    lon, lat, z = syn.particle_cloud(n, seed=seed + 1, three_d=g.z is not None)
    # keep the cloud inside this (smaller) grid
    lon = (g.lon[0] + (lon - 1.0) / 8.2 * g.Lx * 0.8 + 0.1 * g.Lx).astype(np.float32)
    lat = (g.lat[0] + (lat - 55.5) / 4.1 * g.Ly * 0.8 + 0.1 * g.Ly).astype(np.float32)
    if g.z is not None:
        z = (z / 90.0 * abs(g.z.min()) * 1.1).astype(np.float32)     # some below the deepest level
        z[: n // 20] = 0.0                                             # at the surface
        z[n // 20: n // 10] = -0.05                                    # inside the wind-drift layer
    if spill:
        lon[: n // 10] += np.float32(g.Lx)                             # outside coverage -> fallback 0
    readers = [refrun.make_grid_reader(g.lon, g.lat, g.z, times, f3, 'current')]
    f2 = None
    if wind:
        f2 = build_wind(g, n_slabs)
        readers.append(refrun.make_grid_reader(g.lon, g.lat, None, times, f2, 'wind'))
    fs = None
    if stokes:
        fs = build_stokes(g, n_slabs, stokes_hs)
        readers.append(refrun.make_grid_reader(g.lon, g.lat, None, times, fs, 'waves'))
    cfg = {'drift:advection_scheme': scheme, 'drift:vertical_advection': bool(with_w)}
    if stokes:
        cfg['drift:stokes_drift_profile'] = stokes
    else:
        cfg['drift:stokes_drift'] = False
    if diffusivity:
        cfg['environment:constant:horizontal_diffusivity'] = diffusivity
    if wind_drift_depth is not None:
        cfg['drift:wind_drift_depth'] = wind_drift_depth
    for k, v in (noise or {}).items():
        cfg['drift:%s_uncertainty' % k if k != 'current_uniform' else 'drift:current_uncertainty_uniform'] = v
    if mixing:
        cfg['drift:vertical_mixing'] = True
        cfg['vertical_mixing:timestep'] = dt_mix
    if diffusivity_model is not None and diffusivity_model != 'environment_no_reader':
        cfg['vertical_mixing:diffusivitymodel'] = diffusivity_model
    if background_diffusivity is not None:
        cfg['vertical_mixing:background_diffusivity'] = background_diffusivity
    if truncate is not None:
        cfg['drift:truncate_ocean_model_below_m'] = truncate
    if w_at_surface:
        cfg['drift:vertical_advection_at_surface'] = True
    seed_kwargs = {}
    if cdf is not None:
        seed_kwargs['current_drift_factor'] = cdf
    start = syn.T0 + timedelta(seconds=start_offset_s)
    if dt < 0:
        start = times[-1]
    o = refrun.run_oceandrift(readers, lon, lat, z, start, dt, steps, config=cfg,
                              seed_kwargs=seed_kwargs, seed=seed)
    meta = dict(name=name, steps=steps, dt=dt, scheme=scheme, with_w=with_w, wind=wind,
                diffusivity=diffusivity, seed=seed, wind_drift_depth=wind_drift_depth,
                start_offset_s=start_offset_s if dt > 0 else None,
                start_index=None if dt > 0 else len(times) - 1,
                slab_step_s=3600, cdf_is_array=cdf is not None, mixing=mixing, dt_mix=dt_mix, stokes=stokes, noise=noise,
                truncate=truncate, w_at_surface=w_at_surface, diffusivity_model=diffusivity_model,
                background_diffusivity=background_diffusivity)
    out = dict(meta=json.dumps(meta), grid_lon=g.lon, grid_lat=g.lat,
               grid_z=np.zeros(0) if g.z is None else g.z,
               u=f3[CURRENT[0]], v=f3[CURRENT[1]], lon0=lon, lat0=lat, z0=z,
               lon=np.asarray(o.elements.lon, dtype=np.float64),
               lat=np.asarray(o.elements.lat, dtype=np.float64),
               z=np.asarray(o.elements.z))      # float32, or float64 once vertical mixing has touched it
    if with_w:
        out['w'] = f3['upward_sea_water_velocity']
    if mixing and 'ocean_vertical_diffusivity' in f3:
        out['kdiff'] = f3['ocean_vertical_diffusivity']
    if stokes:
        for k, v in fs.items():
            out['stokes__' + k] = v
    if wind:
        out['x_wind'], out['y_wind'] = f2['x_wind'], f2['y_wind']
    if cdf is not None:
        out['cdf'] = np.asarray(cdf, dtype=np.float32)
    assert len(o.elements.lon) == n, 'reference deactivated particles in %s' % name
    path = os.path.join(OUT, 'ref_%s.npz' % name)
    np.savez_compressed(path, **out)
    print('wrote', path, 'max |dlon|', np.abs(out['lon'] - lon).max())


def run_leeway_case(name, g, n, steps, dt, object_type=1, seed=0, capsizing=None):
    """Reference Leeway (opendrift/models/leeway.py) with 2-D current and wind readers."""
    import tempfile
    refrun.setup()
    from opendrift.models.leeway import Leeway
    n_slabs = syn.n_slabs_for(steps, dt)
    times, fc = build_fields(g, n_slabs)
    fw = build_wind(g, n_slabs)
    lon, lat, _ = syn.particle_cloud(n, seed=seed + 1, three_d=False)
    lon = (g.lon[0] + (lon - 1.0) / 8.2 * g.Lx * 0.8 + 0.1 * g.Lx).astype(np.float32)
    lat = (g.lat[0] + (lat - 55.5) / 4.1 * g.Ly * 0.8 + 0.1 * g.Ly).astype(np.float32)
    o = Leeway(loglevel=50, logfile=os.path.join(tempfile.gettempdir(), 'oracle_refrun.log'), seed=seed)
    o.add_reader([refrun.make_grid_reader(g.lon, g.lat, None, times, fc, 'current'),
                  refrun.make_grid_reader(g.lon, g.lat, None, times, fw, 'wind')])
    for k, v in {'general:use_auto_landmask': False, 'environment:constant:land_binary_mask': 0,
                 'general:coastline_action': 'none'}.items():
        o.set_config(k, v)
    if capsizing is not None:            # (wind_threshold, wind_threshold_sigma)
        o.set_config('processes:capsizing', True)
        o.set_config('capsizing:wind_threshold', capsizing[0])
        o.set_config('capsizing:wind_threshold_sigma', capsizing[1])
    o.seed_elements(lon=lon, lat=lat, time=syn.T0 if dt > 0 else times[-1], object_type=object_type,
                    **({'capsized': 1} if (capsizing is not None and dt < 0) else {}))
    o.run(steps=steps, time_step=dt, time_step_output=dt)
    assert len(o.elements.lon) == n
    prop = {k: v for k, v in o.leewayprop[object_type].items() if k not in ('OBJKEY', 'Description')}
    meta = dict(name=name, steps=steps, dt=dt, seed=seed, slab_step_s=3600, object_type=object_type, prop=prop, model='Leeway',
                start_offset_s=0, capsizing=list(capsizing) if capsizing is not None else None)
    path = os.path.join(OUT, 'ref_%s.npz' % name)
    np.savez_compressed(path, meta=json.dumps(meta), grid_lon=g.lon, grid_lat=g.lat, u=fc[CURRENT[0]], v=fc[CURRENT[1]],
                        x_wind=fw['x_wind'], y_wind=fw['y_wind'], lon0=lon, lat0=lat,
                        lon=np.asarray(o.elements.lon), lat=np.asarray(o.elements.lat),
                        orientation=np.asarray(o.elements.orientation), crosswind_slope=np.asarray(o.elements.crosswind_slope),
                        capsized=np.asarray(o.elements.capsized))
    print('wrote', path, 'max |dlon|', np.abs(o.elements.lon - lon).max(), 'jibed', int((o.elements.orientation != np.r_[:n] % 2).sum()))


def dateline_fields(field):
    """The readers' axes and fields of the dateline cases: latitude, the current's and the wind's longitudes, u, v, x_wind, y_wind.
    Pure NumPy: the 'smooth' fixtures do not store their fields, the tests rebuild them here."""
    lat = np.arange(-88, 89).astype(np.float32)
    lon_c = np.arange(0, 360).astype(np.float32)
    lon_w = np.arange(-180, 180).astype(np.float32)
    ny = len(lat)
    if field == 'piecewise':
        u = np.zeros((3, ny, 360), np.float32); v = np.zeros_like(u)
        u[:, :, 0:180] = 1
        u[:, :, 180:] = -1
        xw = np.zeros((3, ny, 360), np.float32); yw = np.zeros_like(xw)
        yw[:, :, 0:180] = 1
        yw[:, :, 180:] = -1
    else:
        lo_c, la = np.meshgrid(np.radians(lon_c.astype(np.float64)), np.radians(lat.astype(np.float64)))
        lo_w, _ = np.meshgrid(np.radians(lon_w.astype(np.float64)), np.radians(lat.astype(np.float64)))
        u = np.stack([(0.8 * np.cos(la) * np.sin(2 * lo_c + 0.3 * k) + 0.2 * np.cos(lo_c)) for k in range(3)]).astype(np.float32)
        v = np.stack([(0.3 * np.sin(3 * lo_c) * np.cos(la) * (1 + 0.1 * k)) for k in range(3)]).astype(np.float32)
        xw = np.stack([(8.0 * np.cos(lo_w + 0.2 * k) * np.cos(la)) for k in range(3)]).astype(np.float32)
        yw = np.stack([(5.0 * np.sin(2 * lo_w) + 1.0 * k) for k in range(3)]).astype(np.float32)
    return lat, lon_c, lon_w, u, v, xw, yw


def run_dateline_case(name, field, seeds_lon, seeds_lat, steps, dt, scheme='euler', wdf=0.1):
    """The reference's tests/readers/test_interpolation.py:43-148 (test_dateline) with in-memory readers: a current
    reader on lon 0..359 (global, 0-360 convention) and a wind reader on lon -180..179 (global, -180-180 convention),
    lat -88..88, daily slabs.  field='piecewise' are the test's own fields (u = +1 east of 0, -1 west; wind v = +1 on
    the western half of its grid, -1 on the eastern); 'smooth' varies with lon / lat so that the seam cells matter."""
    lat, lon_c, lon_w, u, v, xw, yw = dateline_fields(field)
    times = syn.slab_times(3, 86400)
    lon0 = np.asarray(seeds_lon, dtype=np.float32)
    lat0 = np.asarray(seeds_lat, dtype=np.float32)
    n = len(lon0)
    z0 = np.zeros(n, dtype=np.float32)
    readers = [refrun.make_grid_reader(lon_c, lat, None, times, {CURRENT[0]: u, CURRENT[1]: v}, 'current'),
               refrun.make_grid_reader(lon_w, lat, None, times, {'x_wind': xw, 'y_wind': yw}, 'wind')]
    assert readers[0].periodic and readers[1].periodic
    cfg = {'drift:advection_scheme': scheme, 'drift:vertical_advection': False, 'drift:stokes_drift': False}
    o = refrun.run_oceandrift(readers, lon0, lat0, z0, syn.T0, dt, steps, config=cfg, seed_kwargs={'wind_drift_factor': wdf})
    assert len(o.elements.lon) == n, 'reference deactivated particles in %s' % name
    meta = dict(name=name, steps=steps, dt=dt, scheme=scheme, with_w=False, wind=True, diffusivity=0.0, seed=0,
                wind_drift_depth=None, start_offset_s=0, start_index=None, slab_step_s=86400, cdf_is_array=False,
                mixing=False, dt_mix=60.0, stokes=None, noise=None, wdf=wdf, field=field)
    path = os.path.join(OUT, 'ref_%s.npz' % name)
    fields = dict(u=u, v=v, x_wind=xw, y_wind=yw) if field == 'piecewise' else {}       # (the smooth ones would exceed 1 MB)
    np.savez_compressed(path, meta=json.dumps(meta), grid_lon=lon_c, grid_lat=lat, grid_z=np.zeros(0), **fields,
                        wind_lon=lon_w, wind_lat=lat, lon0=lon0, lat0=lat0, z0=z0,
                        lon=np.asarray(o.elements.lon, dtype=np.float64), lat=np.asarray(o.elements.lat, dtype=np.float64),
                        z=np.asarray(o.elements.z))
    print('wrote', path, 'first four', np.asarray(o.elements.lon)[:4], np.asarray(o.elements.lat)[:4])


def dateline_cases():
    rng = np.random.default_rng(42)
    near = np.concatenate([rng.uniform(-1.5, 1.5, 150), rng.uniform(178.5, 181.5, 150)])
    near = (near + 180.0) % 360.0 - 180.0
    lon_a = np.concatenate([[-2, 2, -175, 175], near])
    lat_a = np.concatenate([[60, 60, 60, 60], rng.uniform(-80, 80, 300)])
    run_dateline_case('dateline_piecewise_euler', 'piecewise', lon_a, lat_a, 2, 3600)
    lons, lats = np.meshgrid(np.arange(-180, 181, 20), np.arange(-80, 81, 20))
    run_dateline_case('dateline_piecewise_spread', 'piecewise', lons.ravel(), lats.ravel(), 2, 3600 * 12)
    lon_c = np.concatenate([near, rng.uniform(-180, 180, 400)])
    lat_c = rng.uniform(-85, 85, len(lon_c))
    run_dateline_case('dateline_smooth_rk4', 'smooth', lon_c, lat_c, 6, 3600, scheme='runge-kutta4')
    run_dateline_case('dateline_smooth_euler', 'smooth', lon_c, lat_c, 4, 7200, scheme='euler', wdf=0.03)


def run_gyre_case(name, n, steps, dt, scheme, seed=0, epsilon=0.25, omega=0.628, A=0.25, cdf=None, example=False):
    """BASELINE configs[0]: the reference's analytical double-gyre reader on its stereographic plane
    (examples/example_double_gyre_advection_schemes.py; reader_double_gyre.py), unmodified reference, with
    oracle/proj_stere.py + oracle/geod_karney.py standing in for pyproj."""
    refrun.setup()
    from opendrift.readers import reader_double_gyre
    from opendrift.models.oceandrift import OceanDrift
    rng = np.random.default_rng(seed)
    dg = reader_double_gyre.Reader(epsilon=epsilon, omega=omega, A=A)
    if example:
        x, y = np.array([.6]), np.array([.3])                 # the example's seed point
    else:
        x = rng.uniform(-0.03, 2.03, n)                       # a few per cent start outside the box (fallback 0)
        y = rng.uniform(-0.03, 1.03, n)
    lon, lat = dg.xy2lonlat(x, y)
    o = OceanDrift(loglevel=50, logfile='/tmp/od_gyre.log')
    o.set_config('environment:fallback:land_binary_mask', 0)
    o.set_config('general:use_auto_landmask', False)
    o.set_config('drift:advection_scheme', scheme)
    o.add_reader(dg)
    kw = {}
    if cdf is not None:
        kw['current_drift_factor'] = cdf
    o.seed_elements(lon, lat, time=dg.initial_time, **kw)
    o.run(steps=steps, time_step=dt)
    assert len(o.elements.lon) == len(lon)
    meta = dict(kind='double_gyre', scheme=scheme, dt=dt, steps=steps, epsilon=epsilon, omega=omega, A=A,
                proj4=dg.proj4, initial_time=dg.initial_time.isoformat())
    out = dict(seed_lon=np.asarray(lon, dtype=np.float64), seed_lat=np.asarray(lat, dtype=np.float64),
               lon=np.asarray(o.elements.lon, dtype=np.float64), lat=np.asarray(o.elements.lat, dtype=np.float64),
               meta=json.dumps(meta))
    if cdf is not None:
        out['cdf'] = np.asarray(cdf, dtype=np.float32)
    np.savez_compressed(os.path.join(OUT, 'ref_%s.npz' % name), **out)
    fx, fy = dg.lonlat2xy(o.elements.lon, o.elements.lat)
    print('wrote', name, len(lon), 'x range %.3f..%.3f' % (fx.min(), fx.max()))


def gyre_cases():
    rng = np.random.default_rng(7)
    run_gyre_case('gyre_rk4', 600, 60, 0.1, 'runge-kutta4', seed=1)
    run_gyre_case('gyre_rk2', 600, 40, 0.1, 'runge-kutta', seed=2)
    run_gyre_case('gyre_euler', 600, 40, 0.01, 'euler', seed=3)
    run_gyre_case('gyre_rk4_back_cdf32', 400, 30, -0.1, 'runge-kutta4', seed=4, epsilon=0.1,
                  cdf=rng.uniform(0.5, 1.0, 400).astype(np.float32))
    for scheme, tag in (('euler', 'euler'), ('runge-kutta', 'rk2'), ('runge-kutta4', 'rk4')):
        for dt, dtag in ((0.01, 'dt001'), (0.1, 'dt01')):          # the six runs of the example (duration 6 s)
            run_gyre_case('gyre_example_%s_%s' % (tag, dtag), 1, int(round(6 / dt)), dt, scheme, example=True)


# ---- the BENCHMARKED configurations at 1e5 particles (BASELINE.json configs[1], [3], [4]) ---------------------------------------
# The forcing is syn.* on the full 512 x 512 x 50 grid: it is regenerated by the tests from the same formulas, so the fixtures hold
# only the configuration and the reference's final state (seeds: syn.particle_cloud(n, seed)).
BIG_N = 100_000
BIG_SAMPLE = 30_000        # elements whose final state is stored: a fixed, seeded sample of the BIG_N that run (keeps a fixture < 1 MB)


def big_sample_ids():
    return np.sort(np.random.default_rng(2024).choice(BIG_N, size=BIG_SAMPLE, replace=False)).astype(np.int32)


def big_fields(kind, n_slabs):
    g = syn.GridSpec() if kind != 'cfg5' else syn.GridSpec(nz=1)
    times = syn.slab_times(n_slabs)
    secs = [(t - syn.T0).total_seconds() for t in times]
    uv = [syn.double_gyre_uv(g, s, three_d=g.z is not None) for s in secs]
    out = {'current': {CURRENT[0]: np.stack([a for a, _ in uv]), CURRENT[1]: np.stack([b for _, b in uv])}}
    if kind in ('cfg2', 'cfg4'):
        out['current']['upward_sea_water_velocity'] = np.stack([syn.upward_w(g)] * n_slabs)
    if kind == 'cfg4':
        out['current']['ocean_vertical_diffusivity'] = np.stack([syn.vertical_diffusivity(g, s) for s in secs])
    if kind in ('cfg4', 'cfg5'):
        w = [syn.wind_xy(g, s) for s in secs]
        out['wind'] = {'x_wind': np.stack([a for a, _ in w]), 'y_wind': np.stack([b for _, b in w])}
    if kind == 'cfg4':
        st = [syn.stokes_xy(g, s) for s in secs]
        out['waves'] = {'sea_surface_wave_stokes_drift_x_velocity': np.stack([a for a, _ in st]),
                        'sea_surface_wave_stokes_drift_y_velocity': np.stack([b for _, b in st]),
                        'sea_surface_wave_significant_height': np.stack([syn.wave_height(g, 0.0)] * n_slabs)}
    return g, times, out


BIG = {
    # OceanDrift RK4 + vertical advection on the u/v/w reader (the bench's workload); starts half an hour in, so that the
    # run crosses a reader time step (new slab pair) after three steps
    'cfg2': dict(model='OceanDrift', steps=8, dt=600, start_offset_s=1800, seed=11,
                 config={'drift:advection_scheme': 'runge-kutta4', 'drift:vertical_advection': True, 'drift:stokes_drift': False}),
    # 'OpenOil3D' forcing set: 3-D current + w + K, wind, Stokes drift; vertical mixing + RK4
    'cfg4': dict(model='OceanDrift', steps=4, dt=600, start_offset_s=2400, seed=12,
                 config={'drift:advection_scheme': 'runge-kutta4', 'drift:vertical_advection': True, 'drift:vertical_mixing': True,
                         'vertical_mixing:timestep': 60.0, 'drift:stokes_drift_profile': 'Phillips'}),
    # Leeway, Euler, 2-D current + wind
    'cfg5': dict(model='Leeway', steps=8, dt=600, start_offset_s=1800, seed=13, config={}, object_type=1),
}


def run_big_case(kind):
    c = BIG[kind]
    n_slabs = syn.n_slabs_for(c['steps'], c['dt']) + 1
    g, times, fields = big_fields(kind, n_slabs)
    lon, lat, z = syn.particle_cloud(BIG_N, seed=c['seed'], three_d=g.z is not None)
    readers = [refrun.make_grid_reader(g.lon, g.lat, g.z if nm == 'current' else None, times, f, nm) for nm, f in fields.items()]
    start = syn.T0 + timedelta(seconds=c['start_offset_s'])
    kw = {'object_type': c['object_type']} if c['model'] == 'Leeway' else {}
    o = refrun.run_oceandrift(readers, lon, lat, z if c['model'] != 'Leeway' else 0, start, c['dt'], c['steps'], config=c['config'],
                              seed_kwargs=kw, model=c['model'], seed=0)
    assert len(o.elements.lon) == BIG_N, 'reference deactivated particles in %s' % kind
    ids = big_sample_ids()
    out = dict(meta=json.dumps(dict(kind=kind, n=BIG_N, n_slabs=n_slabs, **{k: v for k, v in c.items()})), ids=ids,
               lon=np.asarray(o.elements.lon, dtype=np.float64)[ids], lat=np.asarray(o.elements.lat, dtype=np.float64)[ids])
    if c['model'] == 'Leeway':
        out['orientation'] = np.asarray(o.elements.orientation).astype(np.int8)[ids]
    else:
        out['z'] = np.asarray(o.elements.z)[ids]
    np.savez_compressed(os.path.join(OUT, 'ref_big_%s.npz' % kind), **out)
    print('wrote ref_big_%s' % kind, 'max |dlon|', np.abs(out['lon'] - lon[ids]).max(), 'z dtype', out.get('z', np.zeros(0)).dtype)


def main():
    import sys
    if 'gyre' in sys.argv[1:]:
        return gyre_cases()
    if 'big' in sys.argv[1:]:
        for kind in [a for a in sys.argv[1:] if a in BIG] or list(BIG):
            run_big_case(kind)
        return
    g3 = syn.GridSpec(nx=40, ny=36, nz=8, lon0=2.0, dlon=0.05, lat0=56.0, dlat=0.03, dz=12.0)
    g2 = syn.GridSpec(nx=40, ny=36, nz=1, lon0=2.0, dlon=0.05, lat0=56.0, dlat=0.03)
    n = 1500
    run_case('rk4_3d', g3, n, 14, 600, 'runge-kutta4')
    run_case('rk2_3d', g3, n, 14, 600, 'runge-kutta')
    run_case('euler_3d', g3, n, 14, 600, 'euler')
    run_case('rk4_2d', g2, n, 14, 600, 'runge-kutta4')
    run_case('rk4_3d_offgrid', g3, n, 8, 900, 'runge-kutta4', spill=True, start_offset_s=450)
    rng = np.random.default_rng(7)
    run_case('rk4_3d_cdf32', g3, n, 8, 600, 'runge-kutta4',
             cdf=rng.uniform(0.5, 1.0, n).astype(np.float32))
    run_case('rk4_3d_backward', g3, n, 8, -600, 'runge-kutta4')
    run_case('rk4_3d_full', g3, n, 10, 600, 'runge-kutta4', with_w=True, wind=True, diffusivity=10.0)
    run_case('euler_2d_wind', g2, n, 10, 600, 'euler', wind=True, wind_drift_depth=0)
    run_case('rk4_3d_noise', g3, 800, 6, 600, 'runge-kutta4', wind=True, diffusivity=5.0,
             noise={'current': 0.1, 'current_uniform': 0.05, 'wind': 1.0})
    run_case('rk2_3d_noise', g3, 800, 5, 600, 'runge-kutta', noise={'current': 0.2})
    run_case('rk4_3d_land', g3, n, 10, 600, 'runge-kutta4', holes=True)
    run_case('euler_2d_land', g2, n, 10, 600, 'euler', holes=True)
    run_leeway_case('leeway_piw1', g2, 1200, 12, 600, object_type=1)
    run_leeway_case('leeway_piw4', g2, 1200, 8, 900, object_type=4, seed=5)
    run_leeway_case('leeway_piw1_capsizing', g2, 1200, 10, 600, object_type=1, seed=2, capsizing=(8.0, 5.0))
    run_case('rk4_3d_stokes_phillips', g3, n, 6, 600, 'runge-kutta4', wind=True, stokes='Phillips')
    run_case('euler_3d_stokes_mono_nohs', g3, n, 6, 600, 'euler', wind=True, stokes='monochromatic', stokes_hs=False)
    run_case('rk2_3d_stokes_exp', g3, n, 5, 600, 'runge-kutta', wind=True, stokes='exponential')
    run_case('rk4_3d_mixing', g3, 600, 7, 600, 'runge-kutta4', mixing=True, dt_mix=60.0)
    run_case('euler_3d_mixing_w', g3, 600, 4, 900, 'euler', mixing=True, dt_mix=100.0, with_w=True)
    dateline_cases()
    run_case('rk4_3d_truncate_wsurf', g3, n, 8, 600, 'runge-kutta4', with_w=True, wind=True, truncate=40.0, w_at_surface=True)
    run_case('rk2_3d_truncate', g3, n, 6, 900, 'runge-kutta', truncate=25.0)
    run_case('rk2_3d_stokes_w', g3, 900, 5, 600, 'runge-kutta', wind=True, stokes='Phillips', with_w=True)
    run_case('rk4_3d_cfg4', g3, 600, 5, 600, 'runge-kutta4', wind=True, stokes='Phillips', mixing=True, dt_mix=60.0, with_w=True)
    run_case('rk4_3d_mixing_large1994', g3, 600, 5, 600, 'runge-kutta4', mixing=True, dt_mix=60.0, wind=True,
             diffusivity_model='windspeed_Large1994')
    run_case('euler_3d_mixing_sundby1983', g3, 600, 4, 900, 'euler', mixing=True, dt_mix=100.0, wind=True,
             diffusivity_model='windspeed_Sundby1983', background_diffusivity=1e-4)
    run_case('rk2_3d_mixing_env_fallback', g3, 600, 4, 600, 'runge-kutta', mixing=True, dt_mix=60.0, wind=True,
             diffusivity_model='environment_no_reader')
    gyre_cases()


if __name__ == '__main__':
    main()
