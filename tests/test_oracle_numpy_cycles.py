"""orc_test_cycles -- the oracle's mg_solve loop run with a fixed sweep schedule, the oracle side of every GPU cycle test at
nrelax values the adaptive solve reaches only when it stalls (tests/test_gpu_cycle_schedule.py) -- against the whole-array
numpy multigrid of tests/test_oracle_numpy_mg.py given the same schedule: the residual after every cycle and the final
stream function, red-black order, closed basin and doubly periodic.  (CPU test, no GPU.)"""
import numpy as np
import pytest

from common import base_kw, periodic_psi, synth_psi
from oracle import oracle as O
from test_oracle_numpy_mg import numpy_solve

SCHEDULE = [2, 5, 9, 17, 3, 4]


@pytest.mark.parametrize("periodic", [False, True], ids=["closed", "periodic"])
@pytest.mark.parametrize("nl", [2, 4, 10])
@pytest.mark.parametrize("N", [32, 64])
def test_cycle_schedule_against_numpy_multigrid(N, nl, periodic):
    kw = base_kw(N, nl, **({"sbc": -1.} if periodic else {}))
    m = O.Model(O.make_params(**kw)); m.set_smoother("rb")
    psi0 = periodic_psi(N, nl) if periodic else synth_psi(N, nl)
    m.set(O.PSI, psi0); m.set_const()
    q = m.get(O.Q)
    strl = m.get(O.STR)[:nl - 1]
    dh = np.array(kw["dh"], dtype=float)
    start = np.zeros_like(psi0)
    m.set(O.PSI, start)
    resa = m.test_cycles(SCHEDULE)
    ref, st, hist = numpy_solve(start, q, strl, dh, kw["L0"], bc=0 if periodic else -1, schedule=SCHEDULE)
    assert hist == SCHEDULE and st["i"] == len(SCHEDULE)
    # no tolerance stop: the last residuals fall to ~1e-9 |q|, where the two sums' round-off (~1e-16 |q|) is more than
    # 1e-8 of the value, hence the absolute floor
    np.testing.assert_allclose(resa, st["resas"], rtol=1e-8, atol=1e-13 * np.abs(q).max())
    got = m.get(O.PSI)
    assert np.abs(got - ref).max() <= (1e-10 if periodic else 1e-11) * np.abs(ref).max()
    # the schedule is not a stopping rule: the residual keeps falling below the solver tolerance
    assert resa[-1] < resa[0]


def test_cycle_schedule_refusals():
    kw = base_kw(32, 2)
    m = O.Model(O.make_params(**kw)); m.set_smoother("rb")
    m.set(O.PSI, synth_psi(32, 2)); m.set_const()
    for bad, mode in (([1], -1), ([101], -1), ([4, 0], -1), ([4], 0), ([4], 2), ([4], -2)):
        with pytest.raises(ValueError):
            m.test_cycles(bad, mode)
    assert m.test_cycles([2, 100]).shape == (2,)
