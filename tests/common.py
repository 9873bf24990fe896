"""Shared helpers of the test-suite: fixture loading and the three ways a fixture can be replayed
(oracle port on CPU, host-compiled device math on CPU, CUDA library on the GPU)."""
import ctypes as C
import glob
import json
import os
import subprocess
import sys
from datetime import timedelta

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from opendrift_b200 import synthetic as syn            # noqa: E402
from opendrift_b200.engine import bracket, draw_uncertainty   # noqa: E402  (pure-Python host logic)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
CUR = ['x_sea_water_velocity', 'y_sea_water_velocity']


def recorded_reference(name, key, run_reference):
    """What the unmodified reference returned for case `key` of the test that stores its results in tests/golden/<name>_ref.npz:
    a dict of arrays.  The tests compare with these recorded results, so that they need neither the reference package nor a
    copy of it.  With OD_WRITE_REFERENCE=1 in the environment, `run_reference()` runs the reference (oracle/refrun.py) and its
    results replace the stored ones."""
    path = os.path.join(GOLDEN, '%s_ref.npz' % name)
    prefix = key + '/'
    if os.environ.get('OD_WRITE_REFERENCE'):
        res = {k: np.asarray(v) for k, v in run_reference().items()}
        kept = {}
        if os.path.exists(path):
            with np.load(path) as d:
                kept = {k: d[k] for k in d.files if not k.startswith(prefix)}
        kept.update({prefix + k: v for k, v in res.items()})
        np.savez_compressed(path, **kept)
        return res
    with np.load(path) as d:
        res = {k[len(prefix):]: d[k] for k in d.files if k.startswith(prefix)}
    assert res, 'no recorded reference result for %s in %s' % (key, path)
    return res


def fixtures():
    """OceanDrift fixtures."""
    return sorted(n for n in (os.path.basename(p)[4:-4] for p in glob.glob(os.path.join(GOLDEN, 'ref_*.npz')))
                  if not n.startswith('leeway') and not n.startswith('gyre') and not n.startswith('big_'))


def leeway_fixtures():
    return sorted(os.path.basename(p)[4:-4] for p in glob.glob(os.path.join(GOLDEN, 'ref_leeway*.npz')))


class LeewayFixture:
    def __init__(self, name):
        d = np.load(os.path.join(GOLDEN, 'ref_%s.npz' % name))
        self.name, self.meta = name, json.loads(str(d['meta']))
        for k in ('grid_lon', 'grid_lat', 'u', 'v', 'x_wind', 'y_wind', 'lon0', 'lat0', 'lon', 'lat', 'orientation',
                  'crosswind_slope'):
            setattr(self, k, d[k])
        self.capsized = d['capsized'] if 'capsized' in d else None
        self.times = syn.slab_times(self.u.shape[0], self.meta['slab_step_s'])
        self.dt, self.steps, self.n, self.start = self.meta['dt'], self.meta['steps'], len(self.lon0), syn.T0
        self.prop = self.meta['prop']


def run_leeway_port(fx):
    from oracle import advect_port as ap, leeway_port as lp
    rc = ap.GridReader(fx.grid_lon, fx.grid_lat, None, fx.times, {CUR[0]: fx.u, CUR[1]: fx.v})
    rw = ap.GridReader(fx.grid_lon, fx.grid_lat, None, fx.times, {'x_wind': fx.x_wind, 'y_wind': fx.y_wind})
    caps = fx.meta.get('capsizing')
    return lp.run_leeway([rc, rw], fx.lon0, fx.lat0, fx.start, fx.dt, fx.steps, fx.prop, seed=fx.meta['seed'],
                         capsizing=tuple(caps) if caps else None)


def _leeway_elements(fx):
    """Seed the per-element coefficients exactly as the reference does (same draws), via the oracle port."""
    from oracle import leeway_port as lp
    np.random.seed(fx.meta['seed'])
    return lp.seed_coefficients(fx.n, fx.prop)


def run_leeway_hostshim(fx):
    lib = hostshim()
    el = _leeway_elements(fx)
    wind = HsField(fx.grid_lon, fx.grid_lat, None, [fx.x_wind, fx.y_wind], fx.times, (float('nan'), float('nan')))
    cur = HsField(fx.grid_lon, fx.grid_lat, None, [fx.u, fx.v], fx.times, (float('nan'), float('nan')))
    lon, lat = fx.lon0.astype(np.float64), fx.lat0.astype(np.float64)
    moving = np.ones(fx.n, dtype=np.int32)
    jp = np.float32(0.04) * np.ones(fx.n)
    capsized = np.zeros(fx.n, dtype=np.uint8)
    t, dt = fx.start, timedelta(seconds=fx.dt)
    for istep in range(fx.steps):
        a = HsLeewayArgs()
        a.g_wind, a.g_cur, a.t_wind, a.t_cur = wind.g, cur.g, wind.pair(t), cur.pair(t)
        a.n, a.lon, a.lat = fx.n, _p(lon), _p(lat)
        a.dw_slope, a.dw_offset, a.dw_eps = _p(el['downwind_slope']), _p(el['downwind_offset']), _p(el['downwind_eps'])
        a.cw_slope, a.cw_offset, a.cw_eps = _p(el['crosswind_slope']), _p(el['crosswind_offset']), _p(el['crosswind_eps'])
        caps = fx.meta.get('capsizing')
        if caps:
            rc, frm = capsize_draws(fx.meta, capsized, fx.dt)                 # drawn before the jibing draws, as the reference does
            a.capsized, a.rand_capsize, a.capsize_on, a.capsize_from = _p(capsized), _p(rc), 1, frm
            a.wind_threshold, a.wind_sigma = caps[0], caps[1]
        rnd = np.random.random(fx.n)
        a.orientation, a.jibe_probability, a.moving, a.rand = _p(el['orientation']), _p(jp), _p(moving), _p(rnd)
        a.dt, a.capsize_fraction, a.pos_f32 = float(fx.dt), 0.4, 1 if istep == 0 else 0
        assert lib.hs_leeway(C.byref(a)) == 0
        t = t + dt
    el['capsized'] = capsized
    return lon, lat, el


def run_leeway_engine(fx, rng='numpy'):
    from opendrift_b200.engine import Engine
    import torch
    eng = Engine(0)
    el = _leeway_elements(fx)
    nan = float('nan')
    wind = eng.add_group(fx.grid_lon, fx.grid_lat, None, 2, fx.times, lambda ti, c: (fx.x_wind, fx.y_wind)[c][ti], (nan, nan))
    cur = eng.add_group(fx.grid_lon, fx.grid_lat, None, 2, fx.times, lambda ti, c: (fx.u, fx.v)[c][ti], (nan, nan))
    lon, lat = eng.to_device(fx.lon0.astype(np.float64)), eng.to_device(fx.lat0.astype(np.float64))
    d = {'dw_slope': eng.to_device(el['downwind_slope']), 'dw_offset': eng.to_device(el['downwind_offset']),
         'dw_eps': eng.to_device(el['downwind_eps']), 'cw_slope': eng.to_device(el['crosswind_slope']),
         'cw_offset': eng.to_device(el['crosswind_offset']), 'cw_eps': eng.to_device(el['crosswind_eps']),
         'orientation': eng.to_device(el['orientation']),
         'capsized': eng.to_device(np.zeros(fx.n, dtype=np.uint8)) if fx.meta.get('capsizing') else None,
         'jibe_probability': eng.to_device(np.float32(0.04) * np.ones(fx.n))}
    ids = eng.to_device(np.arange(fx.n, dtype=np.int32))
    t, dt = fx.start, timedelta(seconds=fx.dt)
    for istep in range(fx.steps):
        kw = {}
        caps = fx.meta.get('capsizing')
        if caps:
            kw = dict(capsizing=(caps[0], caps[1]))
            if rng == 'numpy':
                rc, _ = capsize_draws(fx.meta, d['capsized'].cpu().numpy(), fx.dt)
                kw['rand_capsize'] = eng.to_device(rc)
        rand = eng.to_device(np.random.random(fx.n)) if rng == 'numpy' else None
        eng.leeway_step(wind, cur, t, dt, lon, lat, d, ids=ids, rand=rand, seed=7, step_index=istep, pos_f32=istep == 0, **kw)
        t = t + dt
    eng.sync()
    out = lon.cpu().numpy(), lat.cpu().numpy(), {'orientation': d['orientation'].cpu().numpy(),
                                                  'crosswind_slope': d['cw_slope'].cpu().numpy(),
                                                  'capsized': None if d['capsized'] is None else d['capsized'].cpu().numpy()}
    eng.close()
    return out


class Fixture:
    def __init__(self, name):
        d = np.load(os.path.join(GOLDEN, 'ref_%s.npz' % name))
        self.name = name
        self.meta = json.loads(str(d['meta']))
        self.grid_lon, self.grid_lat = d['grid_lon'], d['grid_lat']
        self.grid_z = d['grid_z'] if d['grid_z'].size else None
        self.w = d['w'] if 'w' in d else None
        if self.meta.get('field') == 'smooth':            # dateline fixtures whose fields are formulas, not stored
            from oracle.make_golden import dateline_fields
            self.u, self.v, self.x_wind, self.y_wind = dateline_fields('smooth')[3:]
        else:
            self.u, self.v = d['u'], d['v']
            self.x_wind = d['x_wind'] if 'x_wind' in d else None
            self.y_wind = d['y_wind'] if 'y_wind' in d else None
        self.wind_lon = d['wind_lon'] if 'wind_lon' in d else self.grid_lon      # the wind reader may have its own grid
        self.wind_lat = d['wind_lat'] if 'wind_lat' in d else self.grid_lat
        self.cdf = d['cdf'] if 'cdf' in d else None
        self.kdiff = d['kdiff'] if 'kdiff' in d else None
        self.stokes = {k[len('stokes__'):]: d[k] for k in d.files if k.startswith('stokes__')} or None
        self.lon0, self.lat0, self.z0 = d['lon0'], d['lat0'], d['z0']
        self.lon, self.lat, self.z = d['lon'], d['lat'], d['z']
        m = self.meta
        self.times = syn.slab_times(self.u.shape[0], m['slab_step_s'])
        self.dt = m['dt']
        self.steps = m['steps']
        self.start = self.times[-1] if self.dt < 0 else syn.T0 + timedelta(seconds=m['start_offset_s'] or 0)
        self.n = len(self.lon0)

    def props(self):
        """Element properties as the reference holds them after release (scalars -> float64 arrays,
        opendrift/elements/elements.py:213-216)."""
        n = self.n
        cdf = self.cdf.astype(np.float32) if self.cdf is not None else np.float32(1) * np.ones(n)
        wdf = np.float32(self.meta.get('wdf', 0.02)) * np.ones(n)
        moving = np.ones(n, dtype=np.int32)
        return cdf, wdf, moving

    def wind_drift_depth(self):
        wdd = self.meta.get('wind_drift_depth')
        return 0.1 if wdd is None else wdd          # OceanDrift default (oceandrift.py:149-152)


def run_port(fx):
    from oracle import advect_port as ap
    f3 = {CUR[0]: fx.u, CUR[1]: fx.v}
    w_own_grid = getattr(fx, 'w_lon', None) is not None          # upward velocity from a reader of its own
    if fx.w is not None and not w_own_grid:
        f3['upward_sea_water_velocity'] = fx.w
    if fx.kdiff is not None:
        f3['ocean_vertical_diffusivity'] = fx.kdiff
    readers = [ap.GridReader(fx.grid_lon, fx.grid_lat, fx.grid_z, fx.times, f3)]
    if fx.w is not None and w_own_grid:
        readers.append(ap.GridReader(fx.w_lon, fx.w_lat, fx.w_z, fx.times, {'upward_sea_water_velocity': fx.w}))
    if fx.x_wind is not None:
        readers.append(ap.GridReader(fx.wind_lon, fx.wind_lat, None, fx.times,
                                     {'x_wind': fx.x_wind, 'y_wind': fx.y_wind}))
    if fx.stokes is not None:
        readers.append(ap.GridReader(fx.grid_lon, fx.grid_lat, None, fx.times, fx.stokes))
    m = fx.meta
    return ap.run_oceandrift(readers, fx.lon0, fx.lat0, fx.z0, fx.start, fx.dt, fx.steps, scheme=m['scheme'],
                             vertical_adv=m['with_w'], wind=m['wind'], wind_drift_depth=fx.wind_drift_depth(),
                             cdf=fx.cdf if fx.cdf is not None else 1.0,
                             wdf=fx.wdf_array if getattr(fx, 'wdf_array', None) is not None else m.get('wdf', 0.02),
                             diffusivity=m['diffusivity'],
                             seed=m['seed'], mixing=m.get('mixing', False), dt_mix=m.get('dt_mix', 60.0),
                             stokes=m.get('stokes'), noise=m.get('noise'), truncate_below=m.get('truncate'),
                             w_at_surface=bool(m.get('w_at_surface')),
                             diffusivity_model={'environment_no_reader': 'windspeed_Large1994'}.get(m.get('diffusivity_model'), m.get('diffusivity_model')),
                             background_diffusivity=1.2e-5 if m.get('background_diffusivity') is None else m['background_diffusivity'])


# ---- host-compiled device math ---------------------------------------------------------------
from opendrift_b200._lib import ProjDesc as _lib_ProjDesc      # noqa: E402


class HsGroup(C.Structure):
    _fields_ = [('ncomp', C.c_int32), ('nx', C.c_int32), ('ny', C.c_int32), ('nz', C.c_int32),
                ('lon_mode', C.c_int32), ('wrap_x', C.c_int32), ('global_x', C.c_int32), ('pad_', C.c_int32),
                ('x0', C.c_double), ('xspan', C.c_double), ('y0', C.c_double), ('yspan', C.c_double),
                ('xmin', C.c_double), ('xmax', C.c_double), ('ymin', C.c_double), ('ymax', C.c_double),
                ('fallback', C.c_float * 2), ('z_levels', C.c_void_p), ('proj', _lib_ProjDesc), ('rotate_vectors', C.c_int32),
                ('pad2_', C.c_int32)]


class HsPair(C.Structure):
    _fields_ = [('tex', C.c_void_p), ('mode', C.c_int32), ('pad_', C.c_int32), ('w', C.c_double)]


class HsLeewayArgsReal(C.Structure):
    _fields_ = [('g_wind', HsGroup), ('g_cur', HsGroup), ('t_wind', HsPair), ('t_cur', HsPair), ('n', C.c_int64),
                ('lon', C.c_void_p), ('lat', C.c_void_p), ('dw_slope', C.c_void_p), ('dw_offset', C.c_void_p),
                ('dw_eps', C.c_void_p), ('cw_slope', C.c_void_p), ('cw_offset', C.c_void_p), ('cw_eps', C.c_void_p),
                ('orientation', C.c_void_p), ('jibe_probability', C.c_void_p), ('moving', C.c_void_p), ('rand', C.c_void_p),
                ('dt', C.c_double), ('capsize_fraction', C.c_float), ('pos_f32', C.c_int32),
                ('capsized', C.c_void_p), ('rand_capsize', C.c_void_p), ('capsize_on', C.c_int32), ('capsize_from', C.c_int32),
                ('wind_threshold', C.c_float), ('wind_sigma', C.c_float)]


HsLeewayArgs = HsLeewayArgsReal


def capsize_draws(meta, capsized, dt):
    """The reference's capsizing draws of one step (leeway.py:443-451) laid out per element: np.random.rand(len(eligible))
    scattered to the eligible elements (capsized == 0 in forward runs, == 1 in backward runs); 2.0 (never selected) elsewhere."""
    frm = 0 if dt >= 0 else 1
    can = np.where(capsized == frm)[0]
    full = np.full(len(capsized), 2.0)
    if len(can) > 0:
        full[can] = np.random.rand(len(can))
    return full, frm


class HsStepArgs(C.Structure):
    _fields_ = [('scheme', C.c_int32), ('factor_f64', C.c_int32), ('pos_f32', C.c_int32), ('z_f64', C.c_int32),
                ('g_uv', HsGroup),
                ('t_start', HsPair), ('t_mid', HsPair), ('t_end', HsPair),
                ('dt', C.c_double), ('n', C.c_int64),
                ('lon', C.c_void_p), ('lat', C.c_void_p), ('z', C.c_void_p),
                ('factor', C.c_void_p), ('moving', C.c_void_p), ('truncate_below', C.c_double),
                ('wind_on', C.c_int32), ('wdf_f64', C.c_int32), ('w_on', C.c_int32), ('w_at_surface', C.c_int32),
                ('g_wind', HsGroup), ('t_wind', HsPair), ('wdf', C.c_void_p), ('wind_drift_depth', C.c_double),
                ('g_w', HsGroup), ('t_w', HsPair), ('z_inout', C.c_void_p),
                ('rand_x', C.c_void_p), ('rand_y', C.c_void_p), ('diffusivity', C.c_void_p),
                ('diffusivity_const', C.c_float), ('z_inout_f64', C.c_int32), ('fast', C.c_int32), ('noise_kinds', C.c_int32),
                ('noise_cur', C.c_void_p), ('noise_wind', C.c_void_p)]


class HsStokesArgs(C.Structure):
    _fields_ = [('n', C.c_int64), ('lon', C.c_void_p), ('lat', C.c_void_p), ('z', C.c_void_p), ('us', C.c_void_p),
                ('vs', C.c_void_p), ('hs', C.c_void_p), ('xwind', C.c_void_p), ('ywind', C.c_void_p),
                ('moving', C.c_void_p), ('dt', C.c_double), ('z_f64', C.c_int32), ('hs_mode', C.c_int32),
                ('profile', C.c_int32), ('pad_', C.c_int32), ('factor', C.c_double), ('d_factor', C.c_void_p), ('factor_f64', C.c_int32),
                ('pad2_', C.c_int32), ('sw_dir', C.c_void_p), ('sw_period', C.c_void_p), ('sw_hs', C.c_void_p), ('ws_dir', C.c_void_p),
                ('ws_period', C.c_void_p), ('ws_hs', C.c_void_p)]

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.factor = 1.0


PROFILES = {'monochromatic': 0, 'exponential': 1, 'Phillips': 2, 'windsea_swell': 3}


def stokes_hs_mode(us, vs, hs, xw, yw):
    """The reference's collective decisions (physics_methods.py:799-812, 893-906): None = no Stokes drift at all,
    else 0 (Hs from the environment), 1 (Hs from wind) or 2 (Hs = 1)."""
    if np.max(np.array(us + vs)) == 0:
        return None
    if hs is not None and hs.max() > 0:
        return 0
    ws = np.sqrt(xw ** 2 + yw ** 2)
    return 1 if ws.max() > 0 else 2


class HsMixArgs(C.Structure):
    _fields_ = [('g', HsGroup), ('t_k', HsPair), ('n', C.c_int64), ('lon', C.c_void_p), ('lat', C.c_void_p),
                ('z_in', C.c_void_p), ('z_out', C.c_void_p), ('moving', C.c_void_p), ('rand', C.c_void_p),
                ('dt_mix', C.c_double), ('sea_floor_const', C.c_double), ('seed', C.c_uint64),
                ('ntimes', C.c_int32), ('z_in_f64', C.c_int32), ('mix_at_surface', C.c_int32), ('pos_f32', C.c_int32),
                ('step_index', C.c_int32), ('model', C.c_int32), ('nlev', C.c_int32), ('pad_', C.c_int32),
                ('wind_speed', C.c_void_p), ('mld_const', C.c_double), ('background', C.c_double), ('k_const', C.c_double)]


MIX_MODEL_IDS = {'windspeed_Large1994': 1, 'environment_no_reader': 1, 'windspeed_Sundby1983': 2}


def mix_model(meta):
    """(id, name) of the analytical diffusivity model of a fixture, or (0, 'environment')."""
    dm = meta.get('diffusivity_model')
    if meta.get('mixing') and dm in MIX_MODEL_IDS:
        return MIX_MODEL_IDS[dm], ('windspeed_Large1994' if dm == 'environment_no_reader' else dm)
    return 0, 'environment'


def z_tolerance(meta, exact=0.0):
    """Depth tolerance of a fixture: `exact` (default: bit for bit) for vertical mixing on profiles that are evaluated with
    elementary arithmetic only; 1e-12 m where the column comes from Large et al. (1994), whose sigma**3 NumPy evaluates
    with its own SIMD pow (an ulp from libm's / CUDA's); 1e-5 m for float32 depths."""
    if not meta.get('mixing'):
        return 1e-5
    return max(exact, 1e-12) if mix_model(meta)[0] == 1 else exact


def mix_background(meta):
    return 1.2e-5 if meta.get('background_diffusivity') is None else meta['background_diffusivity']


_shim = None


def hostshim():
    """Build (once) and load tests/hostshim/libhostshim.so."""
    global _shim
    if _shim is None:
        d = os.path.join(ROOT, 'tests', 'hostshim')
        so, src = os.path.join(d, 'libhostshim.so'), os.path.join(d, 'hostshim.cpp')
        hdrs = glob.glob(os.path.join(ROOT, 'opendrift_b200', 'csrc', '*.cuh')) + glob.glob(os.path.join(ROOT, 'opendrift_b200', 'csrc', '*.inc'))
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in [src] + hdrs):
            subprocess.check_call(['g++', '-O2', '-std=c++17', '-ffp-contract=off', '-shared', '-fPIC',
                                   '-o', so, src])
        _shim = C.CDLL(so)
        _shim.hs_step.restype = C.c_int
    return _shim


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def prep_block(a):
    """What the product does to a reader block before sampling: fill towards the sea floor (host, at block creation)
    and the 10-pass NaN fill (device, od_group_fill_nan) -- emulated here with the oracle's expand_numpy_array."""
    from oracle.advect_port import expand_numpy_array
    a = np.array(a, dtype=np.float32, copy=True)
    if not np.isnan(a).any():
        return a
    if a.ndim == 3:
        for i in range(1, a.shape[0]):
            m = np.isnan(a[i])
            a[i][m] = a[i - 1][m]
    layers = a if a.ndim == 3 else a[None]
    for lay in layers:
        for _ in range(10):
            if not np.isnan(lay).any():
                break
            expand_numpy_array(lay)
    return a


class HsField:
    """A field group for the host shim: builds pair texels with NumPy."""

    def __init__(self, lon, lat, z, comps, times, fallback=(0.0, 0.0)):
        self.lon, self.lat = np.asarray(lon, np.float32), np.asarray(lat, np.float32)
        self.z = None if z is None else np.ascontiguousarray(z, dtype=np.float64)
        self.comps, self.times = comps, times
        g = HsGroup()
        g.ncomp, g.nx, g.ny, g.nz = len(comps), len(self.lon), len(self.lat), 1 if self.z is None else len(self.z)
        from opendrift_b200.engine import grid_geometry
        geo = grid_geometry(self.lon, self.lat)
        g.lon_mode, g.wrap_x, g.global_x = geo['lon_mode'], geo['wrap_x'], geo['global_x']
        g.x0, g.xspan, g.y0, g.yspan = geo['x0'], geo['xspan'], geo['y0'], geo['yspan']
        g.xmin, g.xmax, g.ymin, g.ymax = geo['xmin'], geo['xmax'], geo['ymin'], geo['ymax']
        g.fallback[0], g.fallback[1] = fallback[0], fallback[-1]
        g.z_levels = None if self.z is None else self.z.ctypes.data
        self.g = g
        self._keep = []

    def sample(self, lib, t, lon, lat, z, pos_f32):
        n = len(lon)
        o0, o1 = np.empty(n, np.float32), np.empty(n, np.float32)
        pr = self.pair(t)
        lib.hs_interp(C.byref(self.g), C.byref(pr), C.c_int64(n), _p(lon), _p(lat), _p(z.astype(np.float32)),
                      C.c_int(1 if pos_f32 else 0), _p(o0), _p(o1))
        return o0, o1

    def pair(self, t):
        pr = HsPair()
        br = bracket(self.times, t)
        if br is None:
            pr.mode = 3
            return pr
        ib, ia, w = br
        ja = ib if ia is None else ia
        tex = np.ascontiguousarray(np.stack([prep_block(c[ib]) for c in self.comps] + [prep_block(c[ja]) for c in self.comps],
                                            axis=-1), dtype=np.float32)
        self._keep.append(tex)
        pr.tex, pr.mode, pr.w = tex.ctypes.data, (1 if ia is None else 0), w
        return pr


def run_hostshim(fx, fast=False):
    lib = hostshim()
    m = fx.meta
    cur = HsField(fx.grid_lon, fx.grid_lat, fx.grid_z, [fx.u, fx.v], fx.times)
    wind = HsField(fx.wind_lon, fx.wind_lat, None, [fx.x_wind, fx.y_wind], fx.times) if m['wind'] else None
    wg = (fx.w_lon, fx.w_lat, fx.w_z) if getattr(fx, 'w_lon', None) is not None else (fx.grid_lon, fx.grid_lat, fx.grid_z)
    wfld = HsField(wg[0], wg[1], wg[2], [fx.w], fx.times, (0.0,)) if m['with_w'] else None
    kfld = HsField(fx.grid_lon, fx.grid_lat, fx.grid_z, [fx.kdiff], fx.times, (0.0,)) if m.get('mixing') else None
    sfld = hfld = None
    if m.get('stokes'):
        sfld = HsField(fx.grid_lon, fx.grid_lat, None, [fx.stokes['sea_surface_wave_stokes_drift_x_velocity'],
                                                         fx.stokes['sea_surface_wave_stokes_drift_y_velocity']], fx.times)
        if 'sea_surface_wave_significant_height' in fx.stokes:
            hfld = HsField(fx.grid_lon, fx.grid_lat, None, [fx.stokes['sea_surface_wave_significant_height']], fx.times, (0.0,))
    cdf, wdf, moving = fx.props()
    lon = fx.lon0.astype(np.float64)
    lat = fx.lat0.astype(np.float64)
    z = fx.z0.astype(np.float32).copy()
    np.random.seed(m['seed'])
    t = fx.start
    dt = timedelta(seconds=fx.dt)
    nz_ = m.get('noise') or {}
    for istep in range(fx.steps):
        ncur, nkinds, nwind = draw_uncertainty(fx.n, m['scheme'], nz_.get('current', 0), nz_.get('current_uniform', 0),
                                               nz_.get('wind', 0), with_wind=bool(m['wind']))
        z_new = None
        mix_id, _ = mix_model(m)
        if kfld is not None or mix_id:         # vertical mixing first: it needs the start-of-step positions
            ntimes = abs(int(fx.dt / (m['dt_mix'] * np.sign(fx.dt))))
            rnd = np.ascontiguousarray(np.stack([np.random.random(fx.n) for _ in range(ntimes)]))
            ma = HsMixArgs()
            ma.n = fx.n
            if mix_id:
                xw0, yw0 = wind.sample(lib, t, lon, lat, z, istep == 0)
                ws = np.sqrt(xw0**2 + yw0**2)                                   # PhysicsMethods.wind_speed, float32
                ma.model, ma.nlev, ma.wind_speed = mix_id, len(np.arange(0, np.float32(50) + 2)), _p(ws)
                ma.mld_const, ma.background = 50.0, mix_background(m)
            else:
                ma.g, ma.t_k = kfld.g, kfld.pair(t)
            z_new = np.empty(fx.n, dtype=np.float64)
            ma.lon, ma.lat, ma.z_in, ma.z_out = _p(lon), _p(lat), _p(z), _p(z_new)
            ma.moving, ma.rand = _p(moving), _p(rnd)
            ma.dt_mix, ma.sea_floor_const = m['dt_mix'] * np.sign(fx.dt), 10000.0
            ma.ntimes, ma.z_in_f64 = ntimes, 1 if z.dtype == np.float64 else 0
            ma.pos_f32 = 1 if istep == 0 else 0
            assert lib.hs_mix(C.byref(ma)) == 0
        senv = None
        if sfld is not None:                   # start-of-step environment for the Stokes move
            us, vs = sfld.sample(lib, t, lon, lat, z, istep == 0)
            hs = hfld.sample(lib, t, lon, lat, z, istep == 0)[0] if hfld is not None else None
            xw, yw = wind.sample(lib, t, lon, lat, z, istep == 0)
            senv = (us, vs, hs, xw, yw)
        a = HsStepArgs()
        if ncur is not None:
            ncur = np.ascontiguousarray(ncur)
            a.noise_cur, a.noise_kinds = _p(ncur), nkinds
        if nwind is not None:
            nwind = np.ascontiguousarray(nwind)
            a.noise_wind = _p(nwind)
        a.fast = int(fast)
        a.pos_f32 = 1 if istep == 0 else 0
        a.z_f64 = 1 if z.dtype == np.float64 else 0
        a.scheme = {'euler': 0, 'runge-kutta': 1, 'runge-kutta4': 2}[m['scheme']]
        a.factor_f64 = 1 if cdf.dtype == np.float64 else 0
        a.g_uv = cur.g
        a.t_start, a.t_mid, a.t_end = cur.pair(t), cur.pair(t + dt / 2), cur.pair(t + dt)
        a.dt, a.n = float(fx.dt), fx.n
        a.lon, a.lat, a.z = _p(lon), _p(lat), _p(z)
        a.factor, a.moving = _p(cdf), _p(moving)
        a.truncate_below = float(m.get('truncate') or 0.0)
        if wind is not None:
            a.wind_on, a.wdf_f64, a.g_wind, a.t_wind = 1, (1 if wdf.dtype == np.float64 else 0), wind.g, wind.pair(t)
            a.wdf, a.wind_drift_depth = _p(wdf), fx.wind_drift_depth()
        if wfld is not None:
            if z_new is None and senv is not None:
                z_new = z.copy()          # the Stokes move (after this launch) still needs the start-of-step depth
            zu = z if z_new is None else z_new
            a.w_on, a.g_w, a.t_w, a.z_inout = 1, wfld.g, wfld.pair(t), _p(zu)
            a.w_at_surface = 1 if m.get('w_at_surface') else 0
            a.z_inout_f64 = 1 if zu.dtype == np.float64 else 0
        if m['diffusivity']:
            rx = np.random.normal(scale=1, size=fx.n)
            ry = np.random.normal(scale=1, size=fx.n)
            a.rand_x, a.rand_y, a.diffusivity_const = _p(rx), _p(ry), m['diffusivity']
        assert lib.hs_step(C.byref(a)) == 0
        if senv is not None:
            us, vs, hs, xw, yw = senv
            mode = stokes_hs_mode(us, vs, hs, xw, yw)
            if mode is not None:
                sa = HsStokesArgs()
                sa.n, sa.lon, sa.lat, sa.z = fx.n, _p(lon), _p(lat), _p(z)
                sa.us, sa.vs, sa.hs, sa.xwind, sa.ywind = _p(us), _p(vs), _p(hs), _p(xw), _p(yw)
                sa.moving, sa.dt, sa.z_f64 = _p(moving), float(fx.dt), 1 if z.dtype == np.float64 else 0
                sa.hs_mode, sa.profile = mode, PROFILES[m['stokes']]
                assert lib.hs_stokes(C.byref(sa)) == 0
        if z_new is not None:
            z = z_new
        t = t + dt
    return lon, lat, z


def run_engine(fx, fused=True, sort_every=0, fast=None):
    """Replay a fixture on the GPU through the product Engine (fast=None: the engine's default arithmetic)."""
    import torch
    from opendrift_b200.engine import Engine
    m = fx.meta
    eng = Engine(0)
    three_d = fx.grid_z is not None
    from opendrift_b200.readers.basereader import fill_nan_towards_seafloor

    def cur_supplier(ti, c):                 # host-side block preparation, as StructuredReader.bind does
        a = np.array((fx.u, fx.v)[c][ti], dtype=np.float32, copy=True)
        return fill_nan_towards_seafloor(a) if a.ndim == 3 else a
    cur = eng.add_group(fx.grid_lon, fx.grid_lat, fx.grid_z, 2, fx.times, cur_supplier, (0.0, 0.0))
    wind = wgrp = None
    if m['wind']:
        wind = eng.add_group(fx.wind_lon, fx.wind_lat, None, 2, fx.times,
                             lambda ti, c: (fx.x_wind, fx.y_wind)[c][ti], (0.0, 0.0))
    if m['with_w']:
        wg = (fx.w_lon, fx.w_lat, fx.w_z) if getattr(fx, 'w_lon', None) is not None else (fx.grid_lon, fx.grid_lat, fx.grid_z)
        wgrp = eng.add_group(wg[0], wg[1], wg[2], 1, fx.times, lambda ti, c: fx.w[ti], (0.0,))
    kgrp = None
    if m.get('mixing'):
        kgrp = eng.add_group(fx.grid_lon, fx.grid_lat, fx.grid_z, 1, fx.times, lambda ti, c: fx.kdiff[ti], (0.0,))
    sgrp = hgrp = None
    if m.get('stokes'):
        sx, sy = fx.stokes['sea_surface_wave_stokes_drift_x_velocity'], fx.stokes['sea_surface_wave_stokes_drift_y_velocity']
        sgrp = eng.add_group(fx.grid_lon, fx.grid_lat, None, 2, fx.times, lambda ti, c: (sx, sy)[c][ti], (0.0, 0.0))
        if 'sea_surface_wave_significant_height' in fx.stokes:
            hh = fx.stokes['sea_surface_wave_significant_height']
            hgrp = eng.add_group(fx.grid_lon, fx.grid_lat, None, 1, fx.times, lambda ti, c: hh[ti], (0.0,))
    cdf, wdf, moving = fx.props()
    lon = eng.to_device(fx.lon0.astype(np.float64))
    lat = eng.to_device(fx.lat0.astype(np.float64))
    z = eng.to_device(fx.z0.astype(np.float32)) if three_d or m['wind'] or m['with_w'] else None
    d_cdf, d_wdf, d_mov = eng.to_device(cdf), eng.to_device(wdf), eng.to_device(moving)
    np.random.seed(m['seed'])
    t = fx.start
    dt = timedelta(seconds=fx.dt)
    nz_ = m.get('noise') or {}
    for istep in range(fx.steps):
        first = istep == 0          # element positions are float32 until the first update_positions
        ncur, nkinds, nwind = draw_uncertainty(fx.n, m['scheme'], nz_.get('current', 0), nz_.get('current_uniform', 0),
                                               nz_.get('wind', 0), with_wind=bool(m['wind']))
        d_ncur = eng.to_device(ncur) if ncur is not None else None
        d_nwind = eng.to_device(nwind) if nwind is not None else None
        rand = None
        if m['diffusivity']:
            rand = (eng.to_device(np.random.normal(scale=1, size=fx.n)),
                    eng.to_device(np.random.normal(scale=1, size=fx.n)))
        senv = None
        if sgrp is not None:
            us, vs = eng.interp(sgrp, t, lon, lat, z, pos_f32=first)
            hs = eng.interp(hgrp, t, lon, lat, z, pos_f32=first)[0] if hgrp is not None else None
            xw, yw = eng.interp(wind, t, lon, lat, z, pos_f32=first)
            senv = (us, vs, hs, xw, yw)
        z_new = None
        mix_id, mix_name = mix_model(m)
        if kgrp is not None or mix_id:
            ntimes = abs(int(fx.dt / (m['dt_mix'] * np.sign(fx.dt))))
            rnd = eng.to_device(np.ascontiguousarray(np.stack([np.random.random(fx.n) for _ in range(ntimes)])))
            kw = {}
            if mix_id:
                xw0, yw0 = eng.interp(wind, t, lon, lat, z, pos_f32=first)
                kw = dict(model=mix_name, wind_speed=torch.sqrt(xw0 * xw0 + yw0 * yw0), mld=50.0, background=mix_background(m))
            z_new = eng.vertical_mixing(kgrp, t, lon, lat, z, m['dt_mix'] * np.sign(fx.dt), ntimes, moving=d_mov,
                                        rand=rnd, pos_f32=first, **kw)
        if fused:
            if z_new is None and senv is not None and wgrp is not None:
                z_new = z.clone()         # the Stokes move (after this launch) still needs the start-of-step depth
            eng.step_oceandrift(cur, m['scheme'], t, dt, lon, lat, z if three_d or wind or wgrp else None,
                                factor=d_cdf, moving=d_mov, wind=wind, wdf=d_wdf,
                                wind_drift_depth=fx.wind_drift_depth(), w_group=wgrp, rand=rand,
                                w_at_surface=bool(m.get('w_at_surface')), truncate_below=m.get('truncate'),
                                diffusivity=m['diffusivity'], pos_f32=first, z_update=z_new, fast=fast,
                                noise=d_ncur, noise_kinds=nkinds, wind_noise=d_nwind)
            if senv is not None:
                us, vs, hs, xw, yw = senv
                mode = None
                if eng.minmax(us, vs)[1] != 0:
                    mode = 0 if (hs is not None and eng.minmax(hs)[1] > 0) else (1 if max(eng.minmax(xw)[1], -eng.minmax(xw)[0], eng.minmax(yw)[1], -eng.minmax(yw)[0]) > 0 else 2)
                if mode is not None:
                    eng.stokes_drift(lon, lat, z, us, vs, hs, xw, yw, d_mov, fx.dt, mode, m['stokes'])
            if z_new is not None:
                z = z_new
        else:
            assert not (m['wind'] or m['with_w'] or m['diffusivity'])
            eng.advect_current(cur, m['scheme'], t, dt, lon, lat, z if three_d else None, factor=d_cdf,
                               moving=d_mov, pos_f32=first, fast=fast, noise=d_ncur, noise_kinds=nkinds,
                               truncate_below=m.get('truncate'))
        t = t + dt
    eng.sync()
    out = lon.cpu().numpy(), lat.cpu().numpy(), (z.cpu().numpy() if z is not None else fx.z0)
    eng.close()
    return out


def max_err_deg(lon, lat, rlon, rlat):
    dlon = (lon - rlon + 180.0) % 360.0 - 180.0
    return float(np.max(np.abs(dlon))), float(np.max(np.abs(lat - rlat)))
