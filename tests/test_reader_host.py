"""Reader.get_variables_interpolated at the reader's own precision on the host build of the device sources: bit-equal to the
unmodified reference's StructuredReader (tests/readercases.py)."""
import readercases as rc
from hostengine import HostEngine


def test_reader_output_equals_the_reference_reader_bit_for_bit():
    assert rc.check(HostEngine()) == 27


def test_projected_reader_output_beside_the_live_reference():
    """get_variables_interpolated of readers on conic / stereographic / Mercator planes, with and without the rotation to east /
    north (rotate_to_proj): unrotated values bit-equal, rotated ones to 1e-9 (the rotation angle comes from a differently organised
    inverse geodesic) and float64 like the reference's.  The reference reader's output is recorded in
    tests/golden/reader_proj_ref.npz."""
    import numpy as np
    from datetime import timedelta
    import common
    import projcases as pc
    from opendrift_b200.readers import reader_regular_grid
    eng = HostEngine()
    for case in ('lcc_wgs84_rk4_3d_w', 'stere_wgs84_polar_rk4_3d_w', 'merc_sphere_mixing', 'lcc_sphere_rk2_wind'):
        c, xs, ys, zs, times, fields, lon0, lat0, z0 = pc.setup(case)
        nm = c['readers'][0]
        three_d = nm.startswith('cur3d')
        f = {k: v for k, v in fields[nm].items() if 'velocity' in k and 'upward' not in k}
        rp = reader_regular_grid.Reader(xs, ys, zs if three_d else None, times, f, name=nm, proj4=c['proj4'])
        rp.bind(eng)
        t = times[0] + timedelta(seconds=1000)
        lon, lat, z = lon0.astype(np.float64), lat0.astype(np.float64), z0.astype(np.float64)
        rots = {'plain': None, 'rotated': '+proj=latlong'}

        def reference():
            from oracle import refrun
            rr = refrun.make_grid_reader(xs, ys, zs if three_d else None, times, f, name=nm, proj4=c['proj4'])
            out = {}
            for tag, rot in rots.items():
                b, _ = rr.get_variables_interpolated(list(f), time=t, lon=lon, lat=lat, z=z, rotate_to_proj=rot)
                out.update({'%s_%s' % (tag, k): np.ma.filled(np.ma.masked_invalid(b[k]), np.nan) for k in f})
            return out
        b = common.recorded_reference('reader_proj', case, reference)
        for tag, rot in rots.items():
            a, _ = rp.get_variables_interpolated(list(f), time=t, lon=lon, lat=lat, z=z, rotate_to_proj=rot)
            for k in f:
                x, y = np.ma.filled(np.ma.masked_invalid(a[k]), np.nan), b['%s_%s' % (tag, k)]
                assert x.dtype == y.dtype, (case, rot, k, x.dtype, y.dtype)
                if rot is None:
                    assert np.array_equal(x, y, equal_nan=True)
                else:
                    assert np.nanmax(np.abs(x - y)) < 1e-9


def test_check_arguments_as_reference_style_readers_call_it():
    """variables.py:321-390: get_variables of the reference's gridded readers starts with check_arguments and nearest_time
    (reader_netCDF_CF_generic.py:408-412); a reader written that way runs unchanged on the product's base class, with whole-grid
    and with sub-block requests, and gives what the plain reader gives."""
    import numpy as np
    import pytest
    import common
    from opendrift_b200.readers import reader_regular_grid
    from opendrift_b200.errors import VariableNotCoveredError, OutsideTemporalCoverageError, OutsideSpatialCoverageError
    from datetime import timedelta
    fx = common.Fixture('rk4_2d')
    calls = []

    class Checked(reader_regular_grid.Reader):
        def get_variables(self, requested_variables, time=None, x=None, y=None, z=None):
            requested_variables, time, x, y, z, outside = self.check_arguments(requested_variables, time, x, y, z)
            nearest, *_rest = self.nearest_time(time)
            calls.append((x is None, len(outside)))
            return super().get_variables(requested_variables, nearest, x, y, z)

    fields = {common.CUR[0]: fx.u, common.CUR[1]: fx.v}
    t = fx.times[1] + timedelta(seconds=700)
    lon, lat = fx.lon0[:200].astype(np.float64), fx.lat0[:200].astype(np.float64)
    ref = {}
    for cls, sub in ((reader_regular_grid.Reader, False), (reader_regular_grid.Reader, True), (Checked, False), (Checked, True)):
        r = cls(fx.grid_lon, fx.grid_lat, None, fx.times, fields, name='r', subblocks=sub)
        r.buffer = 3                     # (cells around the requested positions, as set_buffer_size would set it)
        r.bind(HostEngine())
        env, _ = r.get_variables_interpolated(list(fields), time=t, lon=lon, lat=lat, z=np.zeros(200))
        got = {k: np.ma.filled(np.ma.masked_invalid(env[k]), np.nan) for k in fields}
        assert all(np.isfinite(got[k]).all() for k in fields)
        # (a sub-block carries its own float32 axes, so its index arithmetic differs from the whole grid's in the last bits)
        assert all(np.array_equal(got[k], ref.setdefault(sub, got)[k]) for k in fields)
    assert all(np.abs(ref[True][k] - ref[False][k]).max() < 1e-5 for k in fields)
    assert calls and any(c[0] for c in calls) and any(not c[0] for c in calls)
    r = Checked(fx.grid_lon, fx.grid_lat, None, fx.times, fields, name='r')
    with pytest.raises(VariableNotCoveredError):
        r.check_arguments(['x_wind'], fx.times[0], 3.0, 60.0, 0)
    with pytest.raises(OutsideTemporalCoverageError):
        r.check_arguments(list(fields), fx.times[-1] + timedelta(hours=1), 3.0, 60.0, 0)
    with pytest.raises(OutsideSpatialCoverageError):
        r.check_arguments(list(fields), fx.times[0], [50.0, 51.0], [10.0, 11.0], 0)
    v, tt, x, y, z, outside = r.check_arguments(common.CUR[0], None, [float(fx.grid_lon[3]), 99.0], [float(fx.grid_lat[3]), 60.0], None)
    assert v == [common.CUR[0]] and tt == fx.times[0] and list(outside) == [1] and z is None


def test_sub_block_reader_queries_beside_the_live_reference():
    """Reader-level queries on readers that hand out sub-blocks: the block around the positions of the call, the block's own index
    geometry -- bit-equal to the reference's StructuredReader on a reader of the same kind (2-D float32, 3-D float64), whose output
    is recorded in tests/golden/reader_subblock_ref.npz."""
    import numpy as np
    from datetime import timedelta
    import common
    from opendrift_b200.readers import reader_regular_grid
    for fxn in ('rk4_2d', 'rk4_3d'):
        fx = common.Fixture(fxn)
        fields = {common.CUR[0]: fx.u, common.CUR[1]: fx.v}
        t = fx.times[1] + timedelta(seconds=700)
        for sl in (slice(0, 200), slice(200, 230), slice(0, 1500)):
            lon, lat = fx.lon0[sl].astype(np.float64), fx.lat0[sl].astype(np.float64)
            z = np.zeros(len(lon)) if fx.grid_z is None else fx.z0[sl].astype(np.float64)

            def reference():
                from oracle import refrun
                rr = refrun.make_grid_reader(fx.grid_lon, fx.grid_lat, fx.grid_z, fx.times, fields, name='r', subblocks=True)
                rr.buffer = 3
                a, _ = rr.get_variables_interpolated(list(fields), time=t, lon=lon, lat=lat, z=z)
                return {k: np.ma.filled(np.ma.masked_invalid(a[k]), np.nan) for k in fields}
            a = common.recorded_reference('reader_subblock', '%s_%d_%d' % (fxn, sl.start, sl.stop), reference)
            rp = reader_regular_grid.Reader(fx.grid_lon, fx.grid_lat, fx.grid_z, fx.times, fields, name='r', subblocks=True)
            rp.buffer = 3
            rp.bind(HostEngine())
            b, _ = rp.get_variables_interpolated(list(fields), time=t, lon=lon, lat=lat, z=z)
            for k in fields:
                x, y = a[k], np.ma.filled(np.ma.masked_invalid(b[k]), np.nan)
                assert x.dtype == y.dtype and np.array_equal(x, y, equal_nan=True), (fxn, sl, k)
