"""Host-side logic of the product (no GPU): time bracketing, uncertainty draws, element containers, configuration,
reader bookkeeping and the ring-slot residency of field groups -- each against the reference behaviour it mirrors."""
import ctypes as C
from datetime import datetime, timedelta

import numpy as np
import pytest

T0 = datetime(2026, 1, 1)


# ---- time bracketing (variables.py:402-443, structured.py:224-229) --------------------------------------------------
def test_bracket_follows_nearest_time():
    from opendrift_b200.engine import bracket
    times = [T0 + timedelta(hours=i) for i in range(4)]
    assert bracket(times, T0) == (0, None, 0.0)                                   # on a reader time: no after block
    assert bracket(times, T0 + timedelta(hours=2)) == (2, None, 0.0)
    ib, ia, w = bracket(times, T0 + timedelta(minutes=90))
    assert (ib, ia) == (1, 2) and w == 0.5
    ib, ia, w = bracket(times, T0 + timedelta(seconds=3 * 3600 - 1))
    assert (ib, ia) == (2, 3) and w == (3600 - 1) / 3600
    assert bracket(times, times[-1]) == (3, None, 0.0)
    assert bracket(times, T0 - timedelta(seconds=1)) is None                      # covers_time (variables.py:391-400)
    assert bracket(times, times[-1] + timedelta(seconds=1)) is None
    assert bracket([T0], T0 + timedelta(days=3)) == (0, None, 0.0)                # a single time is always valid


def test_port_and_product_agree_on_time_weights():
    from opendrift_b200.engine import bracket
    from oracle import advect_port as ap
    times = [T0 + timedelta(hours=i) for i in range(5)]
    r = ap.GridReader(np.arange(3, dtype=np.float32), np.arange(3, dtype=np.float32), None, times,
                      {'x_wind': np.zeros((5, 3, 3), np.float32)})
    for s in (0, 1, 1799, 3600, 5000, 4 * 3600):
        t = T0 + timedelta(seconds=s)
        tb, ta, ib, ia = r.nearest_time(t)
        br = bracket(times, t)
        assert br[0] == ib
        if t == tb:
            assert br[1] is None
        else:
            assert br[1] == ia and br[2] == (t - tb).total_seconds() / (ta - tb).total_seconds()


# ---- uncertainty draws in the reference's order (environment.py:869-891) --------------------------------------------
def test_uncertainty_draws_follow_the_reference_order():
    from opendrift_b200.engine import draw_uncertainty
    n = 7
    np.random.seed(3)
    cur, kinds, wind = draw_uncertainty(n, 'runge-kutta4', cur_std=0.2, cur_uniform=0.05, wind_std=1.5, with_wind=True)
    np.random.seed(3)
    exp_cur = np.zeros((4, 2, 2, n))
    exp_wind = None
    for stage in range(4):                      # the step's environment, then one call per further RK stage
        exp_cur[stage, 0, 0] = np.random.normal(0, 0.2, n)
        exp_cur[stage, 0, 1] = np.random.normal(0, 0.2, n)
        exp_cur[stage, 1, 0] = np.random.uniform(-0.05, 0.05, n)
        exp_cur[stage, 1, 1] = np.random.uniform(-0.05, 0.05, n)
        if stage == 0:                          # the Runge-Kutta stage calls ask for the current only (physics_methods.py:636-640)
            exp_wind = np.stack([np.random.normal(0, 1.5, n), np.random.normal(0, 1.5, n)])
    assert kinds == 3 and np.array_equal(cur, exp_cur) and np.array_equal(wind, exp_wind)
    assert draw_uncertainty(n, 'euler') == (None, 0, None)


# ---- element containers (elements.py:53-254) ------------------------------------------------------------------------
def test_lagrangian_array_dtypes_and_scalar_promotion():
    from opendrift_b200.elements import LagrangianArray
    a = LagrangianArray(lon=np.array([4.123456789, 5.0]), lat=np.array([60.0, 61.0]), ID=np.array([0, 1]))
    assert a.lon.dtype == np.float32 and a.lat.dtype == np.float32                 # the constructor casts (:156-158)
    assert np.ndim(a.z) == 0 and a.z == 0                                          # defaults stay scalars
    b = LagrangianArray()
    a.move_elements(b, np.array([True, False]))                                    # release: scalars become float64 arrays (:213-216)
    assert len(a) == 1 and len(b) == 1
    assert b.lon.dtype == np.float32 and b.ID[0] == 0 and a.ID[0] == 1
    assert b.z.dtype == np.float64 and b.moving.dtype == np.float64
    c = LagrangianArray(lon=np.array([1.0, 2.0, 3.0]), lat=np.array([1.0, 2.0, 3.0]), ID=np.array([5, 6, 7]))
    d = LagrangianArray()
    c.move_elements(d, np.array([False, True, False]))
    c.move_elements(d, np.array([True, False]))
    assert list(d.ID) == [6, 5] and list(c.ID) == [7]                              # kept / appended in order (:223-228)
    with pytest.raises(TypeError):
        LagrangianArray(lon=np.zeros(2), lat=np.zeros(3))
    with pytest.raises(TypeError):
        LagrangianArray(lon=np.zeros(2), lat=np.zeros(2), no_such_variable=1)


# ---- configuration (config.py:17-119) -------------------------------------------------------------------------------
def test_config_validation_like_the_reference():
    from opendrift_b200.config import Configurable, CONFIG_LEVEL_BASIC
    c = Configurable()
    c._add_config({'a:enum': {'type': 'enum', 'enum': ['x', 'y'], 'default': 'x', 'level': CONFIG_LEVEL_BASIC, 'description': ''},
                   'a:num': {'type': 'float', 'min': 0, 'max': 10, 'default': 1, 'units': '', 'level': CONFIG_LEVEL_BASIC, 'description': ''},
                   'a:flag': {'type': 'bool', 'default': False, 'level': CONFIG_LEVEL_BASIC, 'description': ''}})
    assert c.get_config('a:enum') == 'x' and c.get_config('a:num') == 1
    c.set_config('a:enum', 'y')
    c.set_config('a:num', 2.5)
    assert c.get_config('a:enum') == 'y' and c.get_config('a:num') == 2.5
    with pytest.raises(ValueError):
        c.set_config('a:enum', 'z')
    with pytest.raises(ValueError):
        c.set_config('a:num', 11)
    with pytest.raises(ValueError):
        c.set_config('a:flag', 'yes')
    with pytest.raises(ValueError):
        c.set_config('a:missing', 1)
    with pytest.raises(ValueError):
        c.get_config('a:missing')
    assert c.get_config('a:missing', default=None) is None


# ---- readers --------------------------------------------------------------------------------------------------------
def test_regular_grid_reader_contract():
    from opendrift_b200.readers import reader_regular_grid
    lon, lat = np.linspace(2, 5, 31), np.linspace(60, 57, 41)
    times = [T0 + timedelta(hours=i) for i in range(3)]
    u = np.zeros((3, 4, 41, 31), np.float32)
    r = reader_regular_grid.Reader(lon, lat, [0, -5, -20, -50.0], times, {'x_sea_water_velocity': u, 'y_sea_water_velocity': u})
    assert r.xmin == 2.0 and r.xmax == 5.0 and r.ymin == 57.0 and r.ymax == 60.0 and r.numx == 31 and r.numy == 41
    assert r.start_time == times[0] and r.end_time == times[-1] and r.time_step == timedelta(hours=1)
    assert r.covers_time(times[1]) and not r.covers_time(times[-1] + timedelta(seconds=1))
    ind, x, y = r.covers_positions(np.array([1.0, 3.0, 4.0, 365.0]), np.array([58.0, 58.0, 61.0, 58.0]))
    assert list(ind) == [1, 3] and list(x) == [3.0, 5.0]                          # 365 E is 5 E in the reader's convention
    assert not r.global_coverage()
    blk = r.get_variables(['x_sea_water_velocity'], times[1])
    assert blk['x'].dtype == np.float32 and blk['y'].dtype == np.float32          # reader_netCDF_CF_generic.py:586-587
    assert blk['x_sea_water_velocity'].shape == (4, 41, 31) and list(blk['z']) == [0, -5, -20, -50.0] and blk['time'] == times[1]
    with pytest.raises(NotImplementedError):
        class P(reader_regular_grid.Reader):
            pass
        p = P.__new__(P)
        p.proj4 = '+proj=tmerc +lat_0=0 +lon_0=15 +k_0=0.9996 +ellps=WGS84'            # (stere / merc / lcc are the projections on the GPU path)
        from opendrift_b200.readers.basereader import StructuredReader
        StructuredReader.__init__(p)


# ---- ring-slot residency of a field group -----------------------------------------------------------------------------
class _FakeLib:
    def od_group_define(self, *a):
        return 0


class _FakeEngine:
    """Records what FieldGroup asks of the engine; no CUDA involved."""

    def __init__(self, copy_stream=False):
        self.lib, self.ctx, self.uploads, self.fills = _FakeLib(), None, [], []
        self.dist, self.direction, self.has_copy, self.in_copy, self.on_copy, self.waited = None, 1, copy_stream, False, [], []

    def _check(self, rc):
        assert rc == 0

    def order_after_copies(self):
        pass

    def begin_copy_stream(self):
        if not self.has_copy:
            return False
        self.in_copy = True
        return True

    def end_copy_stream(self):
        self.in_copy = False
        return 'event%d' % len(self.on_copy)

    def wait_event(self, ev):
        self.waited.append(ev)

    def upload(self, gid, slot, comp, data):
        self.uploads.append((slot, comp, int(data[0, 0])))
        if self.in_copy:
            self.on_copy.append((slot, comp, int(data[0, 0])))

    def fill_nan(self, gid, slot, comp, passes):
        self.fills.append((slot, comp, passes))

    def free_group(self, g):
        pass


def test_field_group_ring_residency():
    from opendrift_b200.engine import FieldGroup
    from opendrift_b200 import _lib
    eng = _FakeEngine()
    times = [T0 + timedelta(hours=i) for i in range(6)]
    g = FieldGroup(eng, 0, np.arange(4, dtype=np.float32), np.arange(3, dtype=np.float32), None, 2, times,
                   lambda ti, c: np.full((3, 4), 10 * ti + c, np.float32), (0.0, 0.0), n_slots=3)
    ts, used = g.sample(T0 + timedelta(minutes=30))
    assert ts.mode == _lib.OD_T_LERP and ts.w == 0.5 and used == (0, 1)
    assert sorted(eng.uploads) == [(ts.slot_a, 0, 0), (ts.slot_a, 1, 1), (ts.slot_b, 0, 10), (ts.slot_b, 1, 11)]
    assert len(eng.fills) == 4 and all(f[2] == 10 for f in eng.fills)              # the NaN fill follows every upload
    n_up = len(eng.uploads)
    ts2, _ = g.sample(T0 + timedelta(minutes=45))                                  # same bracket: nothing is uploaded
    assert len(eng.uploads) == n_up and (ts2.slot_a, ts2.slot_b) == (ts.slot_a, ts.slot_b) and ts2.w == 0.75
    ts3, used3 = g.sample(T0 + timedelta(hours=1))                                 # on a reader time: one block only
    assert ts3.mode == _lib.OD_T_FIRST and ts3.slot_a == ts.slot_b and ts3.slot_b == -1 and used3 == (1,)
    ts4, _ = g.sample(T0 + timedelta(minutes=90))                                  # advance: the new slab takes the free slot
    assert ts4.slot_a == ts.slot_b and ts4.slot_b not in (ts.slot_a, ts.slot_b)
    assert len(eng.uploads) == n_up + 2
    ts5, _ = g.sample(T0 + timedelta(minutes=150))                                 # ring is full: the oldest slab is evicted
    assert ts5.slot_a == ts4.slot_b and ts5.slot_b == ts.slot_a
    g.fill_nan = 0
    nf = len(eng.fills)
    g.sample(T0 + timedelta(minutes=210))
    assert len(eng.fills) == nf                                                    # fill switched off
    tsm, usedm = g.sample(times[-1] + timedelta(hours=1))
    assert tsm.mode == _lib.OD_T_MISSING and usedm == ()


def test_field_group_prefetches_the_next_slab_on_the_copy_stream():
    """With a copy stream the slab after the current pair is loaded ahead of time into the free ring slot (backward runs: the
    slab before it); when the run reaches it nothing is uploaded any more, the compute stream just waits for the copy's event."""
    from opendrift_b200.engine import FieldGroup
    eng = _FakeEngine(copy_stream=True)
    times = [T0 + timedelta(hours=i) for i in range(6)]
    g = FieldGroup(eng, 0, np.arange(4, dtype=np.float32), np.arange(3, dtype=np.float32), None, 1, times,
                   lambda ti, c: np.full((3, 4), ti, np.float32), (0.0,), n_slots=3)
    ts, _ = g.sample(T0 + timedelta(minutes=10))
    assert [u[2] for u in eng.uploads] == [0, 1, 2] and [u[2] for u in eng.on_copy] == [2]      # pair on the compute stream, slab 2 ahead
    assert eng.waited == []
    g.sample(T0 + timedelta(minutes=50))
    assert len(eng.uploads) == 3                                                                 # nothing new inside the bracket
    ts2, _ = g.sample(T0 + timedelta(minutes=70))                                                # next bracket: slab 2 is already there
    assert [u[2] for u in eng.uploads] == [0, 1, 2, 3] and [u[2] for u in eng.on_copy] == [2, 3]
    assert eng.waited == ['event1'] and ts2.slot_a == ts.slot_b
    # a step that straddles two brackets pins three slabs: no slot is free, nothing is prefetched, nothing is lost
    g.sample(T0 + timedelta(minutes=110))
    n = len(eng.uploads)
    g.sample(T0 + timedelta(minutes=130), pinned=(1, 2))
    assert len(eng.uploads) == n and g.resident.count(None) == 0
    # backward
    eng2 = _FakeEngine(copy_stream=True)
    eng2.direction = -1
    g2 = FieldGroup(eng2, 0, np.arange(4, dtype=np.float32), np.arange(3, dtype=np.float32), None, 1, times,
                    lambda ti, c: np.full((3, 4), ti, np.float32), (0.0,), n_slots=3)
    g2.sample(T0 + timedelta(minutes=250))
    assert [u[2] for u in eng2.on_copy] == [3]
    g2.prefetch_on = False
    g2.sample(T0 + timedelta(minutes=190))
    assert [u[2] for u in eng2.on_copy] == [3] and len(eng2.uploads) == 3


def test_config_keys_match_the_reference_model_classes():
    """set_config / get_config of a script written for the reference must not raise here: OceanDrift and Leeway expose the
    reference's configuration keys (plus gpu:*), with its defaults except general:coastline_action (no landmask on the GPU
    path: 'none').  The reference's keys and defaults are recorded in tests/golden/config_keys_ref.npz."""
    import json
    import common
    import opendrift_b200.models.oceandrift as po
    import opendrift_b200.models.leeway as pl

    def plain(v):                       # a default as JSON holds it (the recorded form)
        return json.loads(json.dumps(v, default=repr))

    def reference():
        import os
        import tempfile
        from oracle import refrun
        refrun.setup()
        import opendrift.models.oceandrift as ro
        import opendrift.models.leeway as rl
        log = os.path.join(tempfile.gettempdir(), 'od_cfg_test.log')
        return {R.__name__: json.dumps({k: plain(c.get('default')) for k, c in R(loglevel=50, logfile=log)._config.items()})
                for R in (ro.OceanDrift, rl.Leeway)}

    rec = common.recorded_reference('config_keys', 'defaults', reference)

    class NoEngine:
        pass
    for P, extra in ((po.OceanDrift, set()), (pl.Leeway, {'general:seafloor_action', 'seed:seafloor'})):
        r, p = json.loads(str(rec[P.__name__])), P(loglevel=50, engine=NoEngine())
        rk, pk = set(r), set(p._config)
        assert rk - pk == set(), sorted(rk - pk)
        assert {k for k in pk - rk if not k.startswith('gpu:')} == extra
        for k in rk & pk:
            if k != 'general:coastline_action':
                assert r[k] == plain(p._config[k].get('default')), k
    o = po.OceanDrift(loglevel=50, engine=NoEngine())
    o.set_config('general:simulation_name', 'my run')
    o.set_config('seed:z', -5)
    o.set_config('drift:water_column_stretching', True)            # accepted by set_config, refused when the run starts
    o.seed_elements(lon=4, lat=60, time=__import__('datetime').datetime(2026, 1, 1))
    assert o.elements_scheduled.z == -5
    with pytest.raises(NotImplementedError, match='water_column_stretching'):
        o.run(steps=1)
