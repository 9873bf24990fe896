#!/usr/bin/env python
"""bench.py -- particle-steps/s of the RK4 advection hot path (BASELINE.json configs[1]).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one OceanDrift time step (dt = 600 s) of N_local = 10 M particles per GPU: four trilinear +
time interpolations of (u, v) from the synthetic 512x512x50 double-gyre field, three WGS84 geodesic
mid-point moves and the final update_positions -- one launch of step_kernel<RK4> in libodcuda.so.

value  : particle-steps/s with state and forcing slabs resident in HBM (CUDA events, max over ranks)
e2e    : the same steps through the C-ABI with HOST buffers: per step the particle state is copied
         host->device from pinned memory and the new positions device->host; forcing slabs come from
         pinned host memory when the reader time advances
--impl reference : the reference's own CPU algorithm (oracle/advect_port.py, a NumPy/SciPy restatement that
         is bit-identical to the reference on the committed fixtures; /root/reference cannot travel to the
         GPU box) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from datetime import timedelta

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from opendrift_b200 import synthetic as syn  # noqa: E402

DT = 600.0
CUR = ['x_sea_water_velocity', 'y_sea_water_velocity']
METRIC = 'particle-steps/sec (RK4, 10M particles/GPU, 512x512x50 field)'


def measured_peak_hbm():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (one `-lms 10` process, started before the
    warm-up so that the GPU never idles between warm-up and the timed steps; samples are filtered by timestamp)."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '10'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.35)          # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable'], 'samples': 0}
        from datetime import datetime as _dt
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ''
        rows = []
        for line in out.strip().splitlines():
            r = [c.strip() for c in line.split(',')]
            try:
                rows.append((_dt.strptime(r[0], '%Y/%m/%d %H:%M:%S.%f'), float(r[1]), float(r[2]), float(r[3]), r[5:9]))
            except Exception:
                continue
        inside = [r for r in rows if t_begin is not None and t_begin <= r[0] <= t_end]
        window = 'timed region' if inside else 'whole run (no sample fell inside the timed region)'
        sm, mx, pw, reasons = [], [], [], set()
        for ts, a, b, c, flags in (inside or rows):
            sm.append(a)
            mx.append(b)
            pw.append(c)
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], flags):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples'], 'samples': 0}
        # samples under load = those above the idle clock
        load = [x for x in sm if x > 0.5 * max(mx)] or sm
        return {'sm_mhz': float(np.median(load)), 'sm_max_mhz': float(np.max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm), 'samples_under_load': len(load), 'power_w_max': float(np.max(pw)), 'window': window}


PERIOD = 10      # the synthetic double gyre repeats every 36000 s = 10 hourly slabs


class PeriodicSlabs:
    """fields[var][time_index] for a field that is periodic in time: PERIOD distinct slabs serve any run length."""

    def __init__(self, slabs, comp):
        self.slabs, self.comp = slabs, comp

    def __getitem__(self, ti):
        return self.slabs[ti % PERIOD][self.comp]


# ------------------------------------------------------------------------------------------------
def cpu_port_rate(n, steps, seed=123):
    """Reference CPU algorithm (NumPy/SciPy port) on a bounded sample; returns (rate, seconds, threads)."""
    from oracle import advect_port as ap
    grid = syn.GridSpec()
    times = syn.slab_times(syn.n_slabs_for(steps, DT))
    slabs = [syn.double_gyre_uv(grid, (t - syn.T0).total_seconds()) for t in times[:PERIOD]]
    w = syn.upward_w(grid)
    fields = {CUR[0]: PeriodicSlabs(slabs, 0), CUR[1]: PeriodicSlabs(slabs, 1),
              'upward_sea_water_velocity': PeriodicSlabs([(w,)] * PERIOD, 0)}
    reader = ap.GridReader(grid.lon, grid.lat, grid.z, times, fields)
    lon, lat, z = syn.particle_cloud(n, seed=seed)
    t0 = time.perf_counter()
    ap.run_oceandrift([reader], lon, lat, z, syn.T0, DT, steps, scheme='runge-kutta4', vertical_adv=True)
    dt = time.perf_counter() - t0
    return n * steps / dt, dt, 1


def port_reader(n_steps_ahead):
    from oracle import advect_port as ap
    grid = syn.GridSpec()
    times = syn.slab_times(n_steps_ahead)
    slabs = [syn.double_gyre_uv(grid, (t - syn.T0).total_seconds()) for t in times[:PERIOD]]
    w = syn.upward_w(grid)
    fields = {CUR[0]: PeriodicSlabs(slabs, 0), CUR[1]: PeriodicSlabs(slabs, 1),
              'upward_sea_water_velocity': PeriodicSlabs([(w,)] * PERIOD, 0)}
    return ap.GridReader(grid.lon, grid.lat, grid.z, times, fields)


def by_id(torch, state, ids_wanted):
    """(lon, lat, z) NumPy arrays of the elements `ids_wanted` from a device state whose arrays are in cell-sorted order."""
    ids = state['ids'].to(torch.int64)
    inv = torch.empty_like(ids)
    inv[ids] = torch.arange(ids.numel(), device=ids.device)
    pos = inv[torch.as_tensor(ids_wanted, device=ids.device)]
    return tuple(state[k][pos].cpu().numpy() for k in ('lon', 'lat', 'z'))


DUMP_PARTICLES = 2_000_000     # lon, lat (float64) and z (float32) of this many elements over all ranks: 40 MB


def dump_outputs(out_dir, torch, state, rank, world):
    """What the timed steps computed: the final lon / lat / z a caller of the step receives, in element order, as
    out_dir/<name>.npy (a rank suffix per process when there are several).  Above DUMP_PARTICLES / world elements a fixed,
    seeded sample of element ids is written, the same in every run."""
    n, m = state['ids'].numel(), DUMP_PARTICLES // world
    ids = np.arange(n)
    if n > m:
        ids = np.sort(np.random.default_rng(7).choice(n, size=m, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    suffix = '_rank%d' % rank if world > 1 else ''
    for name, a in zip(('lon', 'lat', 'z'), by_id(torch, state, ids)):
        np.save(os.path.join(out_dir, name + suffix + '.npy'), a)


def parity_of_timed_run(eng, torch, st, snap, par_steps, step, args):
    """(a) the last `par_steps` TIMED steps: a subsample of the snapshot taken inside the timed region is advanced by the CPU
    oracle (oracle/advect_port.py, bit-identical to the reference on the committed fixtures) and compared with the positions
    the timed loop produced; (b) 1e5 particles through `--parity-extra` further steps of the same loop (untimed)."""
    from oracle import advect_port as ap
    n = st['ids'].numel()
    rng = np.random.default_rng(2026)
    out = {'tolerance_deg': 1e-6, 'test_bar_deg': 5e-8}
    n_ahead = syn.n_slabs_for(st['k'] + args.parity_extra + 4, DT) + PERIOD
    rd = port_reader(n_ahead)

    def compare(ids, state0, t0, steps, state1, first):
        l0, a0, z0 = by_id(torch, state0, ids)
        c0 = time.perf_counter()
        pl, pa, pz = ap.run_oceandrift([rd], l0, a0, z0, t0, DT, steps, scheme='runge-kutta4', vertical_adv=True, resume=not first)
        secs = time.perf_counter() - c0
        l1, a1, z1 = by_id(torch, state1, ids)
        moved = float(max(np.abs(l1 - l0).max(), np.abs(a1 - a0).max()))
        return {'particles': len(ids), 'steps': steps, 'max_err_deg': float(max(np.abs(l1 - pl).max(), np.abs(a1 - pa).max())),
                'max_err_z_m': float(np.abs(z1.astype(np.float64) - pz.astype(np.float64)).max()), 'max_displacement_deg': moved,
                'cpu_s': secs}
    if snap is not None:
        state0, t0, k0 = snap
        ids = np.sort(rng.choice(n, size=min(n, args.parity_particles), replace=False))
        out['timed_steps'] = compare(ids, state0, t0, par_steps, st, first=(k0 == 0))
        out['timed_steps']['which'] = 'timed steps %d..%d of %d' % (args.steps - par_steps + 1, args.steps, args.steps)
        del state0
    if args.parity_extra > 0:
        state0 = {k: st[k].clone() for k in ('lon', 'lat', 'z', 'ids')}
        t0, k0 = st['t'], st['k']
        for _ in range(args.parity_extra):
            step()
        ids = np.sort(rng.choice(n, size=min(n, 100000), replace=False))
        out['continued_steps'] = compare(ids, state0, t0, args.parity_extra, st, first=(k0 == 0))
        out['continued_steps']['which'] = '%d further steps of the same loop after the timed region' % args.parity_extra
    legs = [out[k] for k in ('timed_steps', 'continued_steps') if k in out]
    out['max_err_deg'] = max(l['max_err_deg'] for l in legs)
    out['max_err_z_m'] = max(l['max_err_z_m'] for l in legs)
    out['ok'] = bool(out['max_err_deg'] < 5e-8 and out['max_err_z_m'] <= 1e-5)
    out['against'] = 'oracle/advect_port.py: NumPy/SciPy restatement of the reference path, bit-identical to the unmodified reference on the committed fixtures (incl. this geometry: tests/golden/ref_big_cfg2.npz)'
    return out


def cpu_reference_rate(n, steps, seed=123):
    """The UNMODIFIED reference (oracle/_ref: a byte-for-byte copy of /root/reference/opendrift made by oracle/build_ref.py, or
    /root/reference itself in the build container) on a bounded sample: OceanDrift.run() of the reference, its own readers base
    class, interpolators and physics; only the third-party packages this image lacks are stubbed (plotting / IO as MagicMock, pyproj by
    oracle/geod_karney.py).  Returns (rate, seconds, threads) or None when the reference package is not there."""
    import tempfile
    from oracle import refrun
    if not refrun.available():
        return None
    refrun.setup()
    from opendrift.models.oceandrift import OceanDrift as RefOceanDrift
    grid = syn.GridSpec()
    times = syn.slab_times(syn.n_slabs_for(steps, DT))
    slabs = [syn.double_gyre_uv(grid, (t - syn.T0).total_seconds()) for t in times[:PERIOD]]
    w = syn.upward_w(grid)
    fields = {CUR[0]: PeriodicSlabs(slabs, 0), CUR[1]: PeriodicSlabs(slabs, 1),
              'upward_sea_water_velocity': PeriodicSlabs([(w,)] * PERIOD, 0)}
    reader = refrun.make_grid_reader(grid.lon, grid.lat, grid.z, times, fields)
    lon, lat, z = syn.particle_cloud(n, seed=seed)
    o = RefOceanDrift(loglevel=50, logfile=os.path.join(tempfile.gettempdir(), 'bench_reference.log'), seed=0)
    o.add_reader(reader)
    for k, v in {'general:use_auto_landmask': False, 'environment:constant:land_binary_mask': 0, 'general:coastline_action': 'none',
                 'drift:advection_scheme': 'runge-kutta4', 'drift:vertical_advection': True, 'drift:stokes_drift': False}.items():
        o.set_config(k, v)
    o.seed_elements(lon=lon, lat=lat, z=z, time=syn.T0)
    t0 = time.perf_counter()
    o.run(steps=steps, time_step=DT, time_step_output=DT)
    dt = time.perf_counter() - t0
    assert o.steps_calculation == steps and len(o.elements.lon) == n
    return n * steps / dt, dt, 1


def cpu_rate(n, steps):
    """(rate, seconds, threads, kind, description): the unmodified reference when its package is present, else the port."""
    r = cpu_reference_rate(n, steps)
    if r is not None:
        return r + ('reference', 'OceanDrift.run() of the UNMODIFIED reference package (oracle/_ref, copied byte for byte from '
                                 '/root/reference/opendrift by oracle/build_ref.py; plotting / IO packages stubbed, pyproj.Geod by '
                                 'oracle/geod_karney.py); single process, single thread, as the reference runs')
    return cpu_port_rate(n, steps) + ('port', 'oracle/advect_port.py = NumPy/SciPy restatement of the reference path, bit-identical to the '
                                              'reference on the committed fixtures (the reference package oracle/_ref is not present)')


def run_reference(args):
    """The reference arm: the reference's own CPU algorithm (single process, as the reference runs) with each
    step a bounded sample of the workload, sized so that K + W steps end within ~2 minutes."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n = args.ref_particles
    if n <= 0:
        budget = 1.2e6                                   # particle-steps (about 90 s at the ~1.3e4 particle-steps/s of the unmodified reference)
        n = int(min(100_000, max(2_000, budget / max(1, args.steps + args.warmup))))
    if args.warmup:
        cpu_rate(n, args.warmup)
    rate, secs, thr, kind, what = cpu_rate(n, args.steps)
    ms = secs * 1e3 / args.steps
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': rate, 'unit': 'particle-steps/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'OceanDrift RK4 + vertical advection, synthetic 512x512x50 double-gyre u/v/w reader, dt=600 s (BASELINE configs[1]); '
                               'CPU arm: each step is a bounded sample of %d particles of that workload' % n},
        'cpu_baseline': {'value': rate, 'unit': 'particle-steps/s', 'cores': thr, 'kind': kind,
                         'sample': '%d particles x %d steps; %s' % (n, args.steps, what)},
        'e2e': {'value': rate, 'unit': 'particle-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------

def configs0_double_gyre(eng, torch, n=10_000_000):
    """BASELINE configs[0] -- the reference's analytical double gyre on its stereographic plane -- as one more measured
    kernel: RK4 launches of od_analytic_advect over n particles (CUDA events, median of 5), one step of a subsample
    checked against the oracle port, and the port's own rate on this host.  Guarded by the caller: it never affects the
    headline line."""
    import time
    from datetime import datetime
    from opendrift_b200.readers import reader_double_gyre
    from oracle import advect_port as ap, gyre_port
    t0 = datetime(2000, 1, 1)
    rd = reader_double_gyre.Reader(initial_time=t0, epsilon=0.25, omega=0.628, A=0.25)
    rd.bind(eng, {v: 0.0 for v in rd.variables})
    d = rd.analytic_desc()
    rng = np.random.default_rng(0)
    lon, lat = rd.xy2lonlat(rng.uniform(0.0, 2.0, n), rng.uniform(0.0, 1.0, n))
    dl0, da0 = eng.to_device(lon), eng.to_device(lat)
    out = []
    for _ in range(5):
        tl, ta = dl0.clone(), da0.clone()
        ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ka.record()
        eng.analytic_advect(d, 'runge-kutta4', (0.0, 0.05, 0.1), 0.1, tl, ta)
        kb.record()
        torch.cuda.synchronize()
        out.append(ka.elapsed_time(kb))
    ms = float(np.median(out))
    m = 20000
    pr = gyre_port.DoubleGyreReader(t0, epsilon=0.25, omega=0.628, A=0.25)
    c0 = time.perf_counter()
    env = ap.get_environment([pr], ['x_sea_water_velocity', 'y_sea_water_velocity'], t0, lon[:m], lat[:m], np.zeros(m))
    pl, pa = ap.advect_ocean_current([pr], 'runge-kutta4', t0, 0.1, lon[:m], lat[:m], np.zeros(m), np.ones(m),
                                     np.ones(m, dtype=np.int32), env)
    cpu_s = time.perf_counter() - c0
    k = 6.371e6 * np.pi / 180
    err = float(np.max(np.hypot((tl[:m].cpu().numpy() - pl) * k, (ta[:m].cpu().numpy() - pa) * k)))
    return {'workload': 'reader_double_gyre on +proj=stere sphere, RK4, dt=0.1 s, %d particles (examples/example_double_gyre_advection_schemes.py at scale)' % n,
            'kernel': 'analytic_step_kernel<RK4, F64, SeriesMath>', 'kernel_ms': ms, 'particle_steps_per_s_kernel': n / (ms * 1e-3),
            'algorithmic_bytes_per_launch': 32 * n, 'hbm_GBps_algorithmic': 32 * n / (ms * 1e-3) / 1e9,
            'bound': 'FP64 / transcendental issue (projection, closed-form field and vector rotation evaluated per stage; no field traffic)',
            'max_err_m_vs_port_one_step': err, 'parity_ok': bool(err < 1e-7),
            'cpu_port_particle_steps_per_s': m / cpu_s, 'cpu_cores': 1}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from opendrift_b200.engine import Engine

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    from opendrift_b200.engine import bind_process_to_gpu_numa
    numa = bind_process_to_gpu_numa(local) if not os.environ.get('OD_BENCH_NONUMA') else {'bound': False, 'off': True}
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    eng = Engine(local)
    dev = eng.device
    n = args.particles
    grid = syn.GridSpec()
    n_times = syn.n_slabs_for(args.warmup + 3 * args.steps + 4, DT) + PERIOD        # (room for the steps after the timed region)
    times = syn.slab_times(n_times)

    # Forcing: rank 0 "reads" the slabs (builds them on the host, keeps them pinned and resident); in a distributed run the other
    # ranks hold NO copy of the data: every new reader time slab reaches their device ring by an NCCL broadcast over NVLink, issued by
    # the field group itself (FieldGroup._load) on the copy stream one slab ahead of the run -- inside the timed loop.
    if world > 1:
        eng.enable_distributed(src=0)
    host_slabs, dev_slabs = [], []
    if rank == 0:
        for ti in range(PERIOD):
            u, v = syn.double_gyre_uv(grid, (times[ti] - syn.T0).total_seconds())
            hu, hv = torch.from_numpy(u).pin_memory(), torch.from_numpy(v).pin_memory()
            host_slabs.append((hu, hv))
            dev_slabs.append((hu.to(dev, non_blocking=True), hv.to(dev, non_blocking=True)))
    torch.cuda.synchronize()
    resident = {'on': True}

    def supplier(ti, c):          # only ever called on the rank that reads
        return dev_slabs[ti % PERIOD][c] if resident['on'] else host_slabs[ti % PERIOD][c]

    grp = eng.add_group(grid.lon, grid.lat, grid.z, 2, times, supplier, (0.0, 0.0), n_slots=3)
    if os.environ.get('OD_BENCH_NOFILL'):
        grp.fill_nan = 0
    if os.environ.get('OD_BENCH_NOPREFETCH'):
        grp.prefetch_on = False
    # upward_sea_water_velocity of the u/v/w reader (static in time)
    h_w = torch.from_numpy(syn.upward_w(grid)).pin_memory() if rank == 0 else None
    d_w = h_w.to(dev) if rank == 0 else None
    wgrp = eng.add_group(grid.lon, grid.lat, grid.z, 1, times, lambda ti, c: d_w if resident['on'] else h_w, (0.0,), n_slots=3)

    # warm cost of the one collective of the design: a slab pair (u, v of one reader time) broadcast from rank 0
    bcast = None
    if world > 1:
        sa = torch.zeros((grid.nz, grid.ny, grid.nx), dtype=torch.float32, device=dev)
        sb = torch.zeros_like(sa)
        for _ in range(3):
            dist.broadcast(sa, 0)
            dist.broadcast(sb, 0)
        torch.cuda.synchronize()
        dist.barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(5):
            dist.broadcast(sa, 0)
            dist.broadcast(sb, 0)
        b1.record()
        torch.cuda.synchronize()
        ms_pair = b0.elapsed_time(b1) / 5
        bcast = {'ms_per_slab_pair_warm': ms_pair, 'bytes_per_slab_pair': 2 * sa.numel() * 4,
                 'GBps': 2 * sa.numel() * 4 / ms_pair / 1e6}
        del sa, sb

    lon0, lat0, z0 = syn.particle_cloud(n, seed=1000 + rank)
    h_lon = torch.from_numpy(lon0.astype(np.float64)).pin_memory()
    h_lat = torch.from_numpy(lat0.astype(np.float64)).pin_memory()
    h_z = torch.from_numpy(z0).pin_memory()
    st = {'lon': h_lon.to(dev), 'lat': h_lat.to(dev), 'z': h_z.to(dev), 't': times[0], 'k': 0,
          'ids': torch.arange(n, dtype=torch.int32, device=dev)}        # element identity travels with the cell sort, as in run()
    dt = timedelta(seconds=DT)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def resort():
        # spatial ordering of the SoA particle arrays (locality of the field gathers); part of the step cost
        perm = eng.sort_by_cell(grp, st['lon'], st['lat'], st['z'])
        for k in ('lon', 'lat', 'z', 'ids'):
            st[k] = eng.permute(perm, st[k])

    step_events = []
    host_us = []

    def step(record=False):
        if args.sort_every and st['k'] % args.sort_every == 0:
            resort()
        if record:
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            h0 = time.perf_counter()
        eng.step_oceandrift(grp, 'runge-kutta4', st['t'], dt, st['lon'], st['lat'], st['z'], w_group=wgrp, pos_f32=(st['k'] == 0))
        if record:
            host_us.append((time.perf_counter() - h0) * 1e6)
            eb.record()
            step_events.append((ea, eb))
        st['t'] += dt
        st['k'] += 1

    # ---- resident run: state and slabs in HBM -----------------------------------------------------------
    # clock ramp: a fresh process on an idle GPU runs its first second ~20 % slow (power state / clock ramp), far
    # longer than W steps of 2 ms; spin the same kernel on scratch copies (simulation state untouched) first
    sampler = ClockSampler(local) if rank == 0 and not os.environ.get('OD_BENCH_NOSMI') else None
    if sampler:
        sampler.start()
    ramp_t0 = time.perf_counter()
    tl, ta, tz = st['lon'].clone(), st['lat'].clone(), st['z'].clone()
    while time.perf_counter() - ramp_t0 < args.ramp_seconds:
        for _ in range(20):
            eng.step_oceandrift(grp, 'runge-kutta4', st['t'], dt, tl, ta, tz, w_group=wgrp)
        torch.cuda.synchronize()
    del tl, ta, tz
    for _ in range(args.warmup):
        step()
    barrier()
    l0 = eng.launches()
    bc0 = eng.dist.slabs_broadcast if eng.dist is not None else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    from datetime import datetime as _dt
    import gc
    gc.collect()
    gc.disable()                       # no collector pauses between launches of the timed steps
    # parity of the TIMED run: the state of every particle at the start of the last `par_steps` timed steps is kept (three
    # device-to-device copies; before the timed region when it covers all K steps) and a subsample is replayed by the CPU oracle
    par_steps = min(args.steps, args.parity_steps)
    snap_at = args.steps - par_steps

    def snapshot():
        return {k: st[k].clone() for k in ('lon', 'lat', 'z', 'ids')}, st['t'], st['k']
    # Exactly K timed steps.  The device time between the steps' own events (end of step j to start of step j + 1) is reported
    # beside the total: a stall of the shared box shows there rather than hiding in the step times.
    del step_events[:]
    del host_us[:]
    snap = snapshot() if snap_at == 0 and not args.no_parity else None
    wall0 = _dt.now()
    e0.record()
    for j in range(args.steps):
        if j == snap_at and j > 0 and not args.no_parity:
            snap = snapshot()
        step(record=True)
    e1.record()
    barrier()
    wall1 = _dt.now()
    ms_total = e0.elapsed_time(e1)
    busy = float(sum(a.elapsed_time(b) for a, b in step_events))
    timed_region = {'ms_total': ms_total, 'ms_in_steps': busy, 'ms_idle_between_steps': ms_total - busy}
    gc.enable()
    launches = eng.launches() - l0
    slabs_bcast = (eng.dist.slabs_broadcast - bc0) if eng.dist is not None else 0
    loop_kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in step_events]))   # includes slab upload / pair packing
    clocks = sampler.stop(wall0, wall1) if sampler else None
    per_step = np.array([a.elapsed_time(b) for a, b in step_events])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, torch, st, rank, world)
    if os.environ.get('OD_BENCH_DEBUG'):          # per-step device times and the gaps between steps, every rank
        gaps = [step_events[k][1].elapsed_time(step_events[k + 1][0]) for k in range(len(step_events) - 1)]
        os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
        json.dump({'rank': rank, 'ms_total': ms_total, 'step_ms': [round(float(x), 3) for x in per_step], 'gap_ms': [round(float(x), 3) for x in gaps],
                   'host_us': [round(float(x), 1) for x in host_us]},
                  open(os.path.join(ROOT, 'gpurun_out', 'steps_n%d_rank%d%s.json' % (world, rank, os.environ.get('OD_BENCH_TAG', ''))), 'w'))

    # dominant kernel alone: CUDA events around single launches of the step kernel on the launching stream
    def kernel_alone(fn):
        out = []
        for _ in range(5):
            ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tl, ta, tz = st['lon'].clone(), st['lat'].clone(), st['z'].clone()
            torch.cuda.synchronize()
            ka.record()
            fn(tl, ta, tz)
            kb.record()
            torch.cuda.synchronize()
            out.append(ka.elapsed_time(kb))
        return float(np.median(out))

    t_now = st['t']
    # The launch is one of two instantiations of the specialised step kernel (csrc/od_spec.cuh): all three time samples between
    # two reader times (4 of the 6 steps of a reader hour), or one of them on a reader time (the step that starts on the hour and
    # the one that ends on it).  kernel_ms is the mean over the six alignments of the hour the timed loop ended in -- the launch
    # mix of the timed loop; the general kernel (OD_OPT_SPEC off, same bits) is timed on the same alignments beside it.
    hour0 = syn.T0 + timedelta(seconds=3600 * int((t_now - syn.T0).total_seconds() // 3600))
    phases = [hour0 + timedelta(seconds=600 * k) for k in range(6)]
    phase_ms = [kernel_alone(lambda tl, ta, tz, tp=tp: eng.step_oceandrift(grp, 'runge-kutta4', tp, dt, tl, ta, tz, w_group=wgrp)) for tp in phases]
    kernel_ms = float(np.mean(phase_ms))
    eng.set_spec(False)
    general_phase_ms = [kernel_alone(lambda tl, ta, tz, tp=tp: eng.step_oceandrift(grp, 'runge-kutta4', tp, dt, tl, ta, tz, w_group=wgrp)) for tp in phases]
    eng.set_spec(True)
    t_now = phases[2]                   # (the variants below: an alignment with all samples between two reader times)
    sort_ms = None
    if args.sort_every:
        sa, sb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        sa.record()
        resort()
        sb.record()
        torch.cuda.synchronize()
        sort_ms = sa.elapsed_time(sb)
    # the operation-by-operation replay of the reference (float32 mid-point azimuths, full Karney geodesic), same launch
    exact_kernel_ms = kernel_alone(lambda tl, ta, tz: eng.step_oceandrift(grp, 'runge-kutta4', t_now, dt, tl, ta, tz, w_group=wgrp, fast=0))
    # the opt-in fast arithmetic (float32 sampling, first-order mid-points), same launch
    fast_kernel_ms = kernel_alone(lambda tl, ta, tz: eng.step_oceandrift(grp, 'runge-kutta4', t_now, dt, tl, ta, tz, w_group=wgrp, fast=1))
    # current advection only (no vertical advection): the plain kernel and its TMA-staged variant (shared-memory field boxes)
    uv_kernel_ms = kernel_alone(lambda tl, ta, tz: eng.advect_current(grp, 'runge-kutta4', t_now, dt, tl, ta, tz))
    eng.set_tile(True)
    tile_kernel_ms = kernel_alone(lambda tl, ta, tz: eng.advect_current(grp, 'runge-kutta4', t_now, dt, tl, ta, tz))
    eng.set_tile(False)

    # ---- parity of what was timed (rank 0; the other ranks wait at the next barrier) ------------------------------------
    parity = None
    if not args.no_parity:
        if rank == 0:
            try:
                parity = parity_of_timed_run(eng, torch, st, snap, par_steps, step, args)
            except Exception as ex:
                parity = {'error': repr(ex)[:300], 'ok': False}
        else:               # the continued steps load new slabs (collectives): every rank takes them, rank 0 alone compares
            for _ in range(args.parity_extra):
                step()

    # ---- the same through OceanDrift.run() on every rank (N > 1) ---------------------------------------------------------------
    api_dist = None
    if world > 1 and not args.no_legs:
        import bench_legs as bl
        try:
            fields = {'current': {CUR[0]: [d[0] for d in dev_slabs], CUR[1]: [d[1] for d in dev_slabs],
                                  'upward_sea_water_velocity': [d_w] * PERIOD}} if rank == 0 else None
            api_dist = bl.leg_api_distributed(eng, torch, dist, n, args.api_steps, fields, grid, rank, world)
        except Exception as ex:
            import traceback
            api_dist = {'error': repr(ex)[:300], 'where': traceback.format_exc()[-500:]}

    # ---- end-to-end: HOST buffers through Engine.advect_current_host, copies inside the timed region -----
    resident['on'] = False
    torch.cuda.synchronize()
    for g_ in (grp, wgrp):                                  # forcing slabs come from pinned host memory again
        g_.resident, g_.ready = [None] * g_.n_slots, [None] * g_.n_slots
    o_lon, o_lat, o_z = torch.empty_like(h_lon).pin_memory(), torch.empty_like(h_lat).pin_memory(), torch.empty_like(h_z).pin_memory()
    e2e_steps = max(3, min(args.steps, 20))
    t_e2e = times[0]
    bufs = [(h_lon, h_lat, h_z), (o_lon, o_lat, o_z)]

    def e2e_step(i, t):
        src, dst = bufs[i % 2], bufs[(i + 1) % 2]
        eng.step_oceandrift_host(grp, 'runge-kutta4', t, dt, src[0], src[1], src[2], dst[0], dst[1], dst[2], w_group=wgrp,
                                 chunks=args.e2e_chunks)

    for i in range(2):
        e2e_step(i, t_e2e)
        t_e2e += dt
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for i in range(e2e_steps):
        e2e_step(i, t_e2e)
        t_e2e += dt
    g1.record()
    barrier()
    e2e_ms = g0.elapsed_time(g1)

    # the same call with PAGEABLE NumPy arrays -- what a caller who holds the reference's element arrays would pass; the driver
    # stages pageable memory itself, so the copies neither overlap each other nor the kernel (reported beside the pinned number)
    e2e_pageable = None
    if world == 1 and not os.environ.get('OD_BENCH_NO_PAGEABLE'):      # (single process only: further steps mean further slab loads,
                                                                          #  which are collectives in a distributed run)
        try:
            pa = [np.array(h_lon.numpy(), copy=True), np.array(h_lat.numpy(), copy=True), np.array(h_z.numpy(), copy=True)]
            pb = [np.empty_like(a) for a in pa]
            pbufs = [pa, pb]
            tp = t_e2e
            psteps = 3
            for i in range(1 + psteps):
                if i == 1:
                    torch.cuda.synchronize()
                    w0 = time.perf_counter()
                src, dst = pbufs[i % 2], pbufs[(i + 1) % 2]
                eng.step_oceandrift_host(grp, 'runge-kutta4', tp, dt, src[0], src[1], src[2], dst[0], dst[1], dst[2], w_group=wgrp,
                                         chunks=args.e2e_chunks)
                tp += dt
            torch.cuda.synchronize()
            pms = (time.perf_counter() - w0) * 1e3 / psteps
            e2e_pageable = {'value': n / (pms * 1e-3), 'unit': 'particle-steps/s', 'ms_per_step': pms, 'steps': psteps,
                            'note': 'pageable NumPy lon / lat / z in and out (rank 0, wall clock around the blocking calls)'}
            del pa, pb
        except Exception as exc:
            e2e_pageable = {'error': repr(exc)[:200]}

    # the link the end-to-end number lives on: this step's bytes (20 B in, 20 B out per particle) as two plain pinned
    # copies running concurrently on two streams
    pcie = None
    if rank == 0:
        try:
            s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
            d_in, d_out = torch.empty_like(h_lon, device=dev), torch.empty_like(h_lat, device=dev)
            d_in2, d_z2 = torch.empty_like(h_lat, device=dev), torch.empty_like(h_z, device=dev)
            torch.cuda.synchronize()
            pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 4
            pa.record()
            for _ in range(reps):
                with torch.cuda.stream(s_in):
                    s_in.wait_event(pa)
                    d_in.copy_(h_lon, non_blocking=True)
                    d_in2.copy_(h_lat, non_blocking=True)
                    d_z2.copy_(h_z, non_blocking=True)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(pa)
                    o_lon.copy_(d_out, non_blocking=True)
                    o_lat.copy_(d_in, non_blocking=True)
                    o_z.copy_(d_z2, non_blocking=True)
            torch.cuda.current_stream().wait_stream(s_in)
            torch.cuda.current_stream().wait_stream(s_out)
            pb.record()
            torch.cuda.synchronize()
            pms = pa.elapsed_time(pb) / reps
            pcie = {'ms_per_step_copies_only': pms, 'particle_steps_per_s_ceiling': n / (pms * 1e-3),
                    'GBps_both_directions': n * 40 / pms / 1e6}
            del d_in, d_out, d_in2, d_z2
        except Exception as exc:        # the probe is informative only
            pcie = {'error': str(exc)}

    if world > 1:       # device-timed, max over ranks
        tt = torch.tensor([ms_total, e2e_ms, kernel_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, e2e_ms, kernel_ms = [float(x) for x in tt.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = n * world * args.steps / (ms_total * 1e-3)
    e2e_value = n * world * e2e_steps / (e2e_ms * 1e-3)
    peak, peak_src = measured_peak_hbm()
    field_bytes = 2 * 3 * grid.nx * grid.ny * grid.nz * 4           # two time slabs x (u, v, w) float32
    state_bytes = 52                                                  # lon, lat read + written (32), z, moving, factor (12), z updated (8)
    b_alg = state_bytes * n + field_bytes                             # SURVEY.md 8(d): 83.5 B per particle-step at 10 M with w
    achieved = b_alg / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, 'profiles', 'step_kernel_traffic.json')
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get('dram_bytes_per_launch')
        except Exception:
            pass
    cpu = None
    if not args.no_cpu:
        rate, secs, thr, kind, what = cpu_rate(args.cpu_particles, args.cpu_steps)
        cpu = {'value': rate, 'unit': 'particle-steps/s', 'cores': thr, 'kind': kind,
               'sample': '%d particles x %d steps (%.1f s) of the same workload: %s' % (args.cpu_particles, args.cpu_steps, secs, what)}
        if kind == 'reference':          # the port beside it, for continuity with round 1
            prate, psecs, _ = cpu_port_rate(args.cpu_particles, 2)
            cpu['port_value'] = prate
    extra = {}
    if world == 1 and not args.no_legs:
        import bench_legs as bl
        for key, fn in (('api', lambda: bl.leg_api(eng, torch, n, args.api_steps,
                                                   {'current': {CUR[0]: [d[0] for d in dev_slabs], CUR[1]: [d[1] for d in dev_slabs],
                                                                'upward_sea_water_velocity': [d_w] * PERIOD}}, grid, peak)),
                        ('cfg4_mixing_wind_stokes', lambda: bl.leg_cfg4(eng, torch, args.cfg4_particles, 40, peak)),
                        ('cfg5_leeway', lambda: bl.leg_cfg5(eng, torch, args.cfg5_particles, 60, peak))):
            try:
                torch.cuda.empty_cache()
                extra[key] = fn()
            except Exception as ex:          # never let a secondary leg touch the headline
                import traceback
                extra[key] = {'error': repr(ex)[:300], 'where': traceback.format_exc()[-400:]}
    gyre = None
    if world == 1 and not os.environ.get('OD_BENCH_NO_GYRE'):
        try:
            gyre = configs0_double_gyre(eng, torch, min(n, 10_000_000))
        except Exception as ex:          # never let the extra measurement touch the headline
            gyre = {'error': repr(ex)[:300]}
    line = {
        'metric': METRIC, 'value': value, 'unit': 'particle-steps/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'OceanDrift RK4 + vertical advection, synthetic 512x512x50 double-gyre u/v/w reader, %d particles per GPU, '
                               'dt=600 s (BASELINE configs[1]%s)' % (n, '; configs[2] sharding' if world > 1 else ''),
                   'particles_per_gpu': n, 'field': '512x512x50 f32 u,v (hourly slabs) + w', 'scheme': 'runge-kutta4',
                   'sort_every': args.sort_every, 'sort_ms': sort_ms, 'clock_ramp_s': args.ramp_seconds, 'mode': 'default arithmetic OD_MATH_SERIES: bit-exact field sampling (float64 index and weight arithmetic of the reference), '
                           'float64 short-arc series geodesic (round-off accurate, full Karney solution beyond its range)',
                   'parallelism': ('particle-index shards x%d, forcing read by rank 0 only and broadcast (NCCL) into the other ranks\' device '
                                   'ring on the copy stream, one slab ahead of the run: %d slab broadcasts INSIDE the timed region; warm cost '
                                   '%.2f ms per 210 MB slab pair = %.0f GB/s' % (world, slabs_bcast, bcast['ms_per_slab_pair_warm'], bcast['GBps']))
                                  if world > 1 else 'single GPU',
                   'l2': 'inputs larger than L2 (state %.0f MB + forcing %.0f MB per step)' % (n * 20 / 1e6, field_bytes / 1e6)},
        'clocks': clocks,
        'timed_region': timed_region,
        'comm': {'slab_broadcasts_in_timed_region': slabs_bcast, 'broadcast': bcast, 'numa': numa,
                 'slab_broadcast_communicator_max_ctas': getattr(eng.dist, 'bcast_ctas', None)} if world > 1 else {'numa': numa},
        'e2e': {'value': e2e_value, 'unit': 'particle-steps/s', 'h2d_bytes_per_step': n * 20, 'd2h_bytes_per_step': n * 20,
                'steps': e2e_steps, 'api': 'od_step_oceandrift_host through Engine.step_oceandrift_host (pinned host lon/lat/z in and out, %d-chunk '
                       'three-stream copy/compute pipeline inside the C-ABI call)' % args.e2e_chunks,
                'pcie_probe': pcie, 'pageable_numpy': e2e_pageable},
        'gpu_launches': launches,
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic, 'peak_source': peak_src, 'kernel': 'step_spec_kernel<RK4, F64, EXTRAS=2> (current advection + vertical advection in one launch; csrc/od_spec.cuh)', 'kernel_ms': kernel_ms,
                     'kernel_ms_by_alignment': phase_ms, 'general_kernel_ms_by_alignment': general_phase_ms, 'general_kernel_ms': float(np.mean(general_phase_ms)),
                     'kernel_ms_mean_in_timed_loop': loop_kernel_ms,
                     'loop_ms_p50': float(np.median(per_step)), 'loop_ms_p95': float(np.percentile(per_step, 95)),
                     'loop_ms_first20_mean': float(per_step[:20].mean()), 'host_us_per_launch_median': float(np.median(host_us)), 'host_us_per_launch_max': float(np.max(host_us)),
                     'algorithmic_bytes_per_launch': b_alg,
                     'note': 'this float64 kernel is bound by FP64 issue (the reference samples its float32 fields with float64 '
                             'index and weight arithmetic, reproduced bit for bit), not by its 65 algorithmic bytes per '
                             'particle-step; see DESIGN.md and profiles/'},
        'cpu_baseline': cpu,
        'parity': parity,
        'api': extra.get('api') if world == 1 else api_dist,
        'cfg4_mixing_wind_stokes': extra.get('cfg4_mixing_wind_stokes'),
        'cfg5_leeway': extra.get('cfg5_leeway'),
        'configs0_double_gyre': gyre,
        'current_only': {'kernel_ms': uv_kernel_ms, 'particle_steps_per_s_kernel': n / (uv_kernel_ms * 1e-3),
                         'note': 'od_advect_current alone (u/v sampling and moves, no vertical advection), same particles'},
        'tma_tile': {'kernel_ms': tile_kernel_ms, 'note': 'opt-in OD_OPT_TILE for current_only: one cp.async.bulk.tensor.4d box per block; same bits; '
                                                          'not faster than L1-served gathers on sorted particles (see DESIGN.md)'},
        'exact_replay_mode': {'kernel_ms': exact_kernel_ms, 'particle_steps_per_s_kernel': n / (exact_kernel_ms * 1e-3),
                              'note': 'OD_MATH_EXACT: the reference arithmetic operation by operation (float32 mid-point azimuth and '
                                      'distance, order-6 Karney geodesic for every move); ~1e-9 deg per step from the default, the size '
                                      'of the reference\'s own float32 arctan2 noise'},
        'fast_mode': {'kernel_ms': fast_kernel_ms, 'particle_steps_per_s_kernel': n / (fast_kernel_ms * 1e-3),
                      'hbm_frac_algorithmic': b_alg / (fast_kernel_ms * 1e-3) / 1e9 / peak,
                      'note': 'opt-in FastMath (float32 sampling, mid-latitude moves on float64 positions), <= 2e-8 deg from the '
                              'reference on the fixtures; not the headline: value/e2e use the default mode'},
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=300)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--particles', type=int, default=10_000_000)
    ap.add_argument('--sort-every', type=int, default=20)
    ap.add_argument('--e2e-chunks', type=int, default=12)
    ap.add_argument('--ramp-seconds', type=float, default=1.5)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--cpu-particles', type=int, default=50_000)
    ap.add_argument('--cpu-steps', type=int, default=4)
    ap.add_argument('--ref-particles', type=int, default=0, help='0 = sized from --steps')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--parity-steps', type=int, default=20, help='timed steps replayed by the CPU oracle (the last ones)')
    ap.add_argument('--parity-particles', type=int, default=20000)
    ap.add_argument('--parity-extra', type=int, default=5, help='further steps after the timed region, replayed for 1e5 particles')
    ap.add_argument('--no-legs', action='store_true', help='skip the api / cfg 4 / cfg 5 legs')
    ap.add_argument('--api-steps', type=int, default=120, help='steps of the OceanDrift.run() leg')
    ap.add_argument('--cfg4-particles', type=int, default=5_000_000)
    ap.add_argument('--cfg5-particles', type=int, default=20_000_000)
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the positions the timed steps computed to DIR/<name>.npy '
                                                          '(--impl b200 only: the reference arm has no such steps)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200 only')
    if args.warmup < 3 and args.impl == 'b200':
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
