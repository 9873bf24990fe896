"""The benchmarked configurations at 1e5 particles (tests/bigcases.py) WITHOUT a GPU: the drop-in model classes on the host build
of the device sources (tests/hostengine.py) against the unmodified reference's results, and the oracle port against the same
results on a subsample (particles are independent in cfg 2).  The GPU run of the same cases is tests/test_zz_gpu_big.py."""
import numpy as np
import pytest

import bigcases as bc
import common
from hostengine import HostEngine


@pytest.fixture()
def host_engine(monkeypatch):
    eng = HostEngine()
    import opendrift_b200.engine as E
    import opendrift_b200.models.basemodel as B
    monkeypatch.setattr(E, 'default_engine', lambda device=None: eng)
    monkeypatch.setattr(B, 'default_engine', lambda device=None: eng)
    yield eng


_cases = {}


def _case(kind):
    if kind not in bc.KINDS:
        pytest.skip('tests/golden/ref_big_%s.npz not generated' % kind)
    if kind not in _cases:
        _cases.clear()
        _cases[kind] = bc.BigCase(kind)
    return _cases[kind]


@pytest.mark.parametrize('kind,sort,ztol', [('cfg2', 20, 0.0), ('cfg2', 0, 0.0), ('cfg5', 20, 0.0), ('cfg4', 0, 1e-9), ('cfg4', 20, 1e-9)])
def test_benchmarked_configuration_on_the_host_build(kind, sort, ztol, host_engine):
    c = _case(kind)
    o = c.model(**{'gpu:sort_interval_steps': sort})
    o.run(steps=c.steps, time_step=c.dt, time_step_output=c.steps * c.dt)
    res = c.check(o, z_tol=ztol)
    assert res['max_err_deg'] < 2e-8


def test_port_matches_reference_on_cfg2_subsample():
    """oracle/advect_port.py (the CPU baseline of bench.py) on the first 4000 stored particles of cfg 2."""
    from oracle import advect_port as ap
    c = _case('cfg2')
    m = 4000
    s = c.ref['ids'][:m]
    f = c.fields['current']
    rd = ap.GridReader(c.grid.lon, c.grid.lat, c.grid.z, c.times, f)
    lon, lat, z = ap.run_oceandrift([rd], c.lon0[s], c.lat0[s], c.z0[s], c.start, c.dt, c.steps, scheme='runge-kutta4', vertical_adv=True)
    assert np.array_equal(lon, c.ref['lon'][:m]) and np.array_equal(lat, c.ref['lat'][:m]) and np.array_equal(z, c.ref['z'][:m])
