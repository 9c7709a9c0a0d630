"""Whole timesteps of the doubly periodic domain (sbc = -1, msqg/qg.h:80, :842-846) -- deterministic, and the
-D_STOCHASTIC=1 build (qg_stochastic.h) with libc rand() noise -- restated in numpy and run beside the C oracle
(red-black order).  The restatement is that of tests/test_oracle_numpy_step.py with every ghost ring wrapped
(np.pad(..., mode="wrap")) and the periodic multigrid solve (numpy_solve(..., bc=0)): same dt sequence, same cycle
counts, q and psi equal to round-off.  So far only the periodic inversion had a numpy pin; this pins the periodic
right-hand side, the dt chain and the stochastic stage updates as well.  (CPU test, no GPU.)"""
import ctypes as C

import numpy as np
import pytest

from common import base_kw, periodic_psi
from oracle import oracle as O
from test_oracle_numpy_mg import numpy_solve
from test_oracle_numpy_rhs import jac, lap, pad, sh, stretch
from test_oracle_numpy_step import NumpyModel, NumpyStochasticModel

WRAP = 0   # pad(): periodic ghost ring


class PeriodicNumpyModel(NumpyModel):
    """NumpyModel on the doubly periodic domain; stochastic=True gives the qg_stochastic.h right-hand side (no
    J(psi, zeta) in the top layer, no J(psi_l, psi_l+1), relaxation -q/tr_stoch)"""

    def __init__(self, kw, psi, stochastic=False):
        super().__init__(kw, psi)
        self.stochastic = stochastic
        P = [pad(psi[l], WRAP) for l in range(self.nl)]
        self.q = np.array([lap(P[l], self.D) for l in range(self.nl)]) + stretch(psi, list(self.s), self.idh0, self.idh1)

    def update(self, q, dtmax):
        kw, nl, D = self.kw, self.nl, self.D
        self.psi, st, _ = numpy_solve(self.psi, q, self.s, self.dh, self.L0, bc=WRAP)     # invertq: warm start
        self.cycles += st["i"]
        P = [pad(self.psi[l], WRAP) for l in range(nl)]
        zeta = np.array([lap(P[l], D) for l in range(nl)])
        Z = [pad(zeta[l], WRAP) for l in range(nl)]
        jd = [jac(P[l], P[l + 1], D) for l in range(nl - 1)]
        dq = np.zeros_like(q)
        for l in range(nl):
            t = kw["beta"] * (sh(P[l], -1, 0) - sh(P[l], 1, 0)) / (2 * D)
            if not (self.stochastic and l == 0):
                t = jac(P[l], Z[l], D) + t
            if not self.stochastic:
                if l > 0:
                    t = t + self.s[l - 1] * (-jd[l - 1]) * self.idh0[l]
                if l < nl - 1:
                    t = t + self.s[l] * jd[l] * self.idh1[l]
            dq[l] = t
        if self.stochastic:
            dq += -q / kw["tr_stoch"]
        tmp = np.array([lap(Z[l], D) for l in range(nl)])
        T = [pad(tmp[l], WRAP) for l in range(nl)]
        dq += self.iRe4 * stretch(tmp, list(self.s), self.idh0, self.idh1) + self.iRe4 * np.array([lap(T[l], D) for l in range(nl)])
        dq[-1] -= kw["Ekb"] / (kw["Rom"] * 2 * self.dh[-1]) * zeta[-1]
        dq[0] -= self.wind
        CFL = kw["CFL"]
        for l in range(nl):
            Pl = P[l]; n = self.N
            ux = -0.25 * (Pl[2:n + 2, 1:n + 2] - Pl[0:n, 1:n + 2] + Pl[2:n + 2, 0:n + 1] - Pl[0:n, 0:n + 1]) / D
            uy = 0.25 * (Pl[1:n + 2, 2:n + 2] - Pl[1:n + 2, 0:n] + Pl[0:n + 1, 2:n + 2] - Pl[0:n + 1, 0:n]) / D
            for u in (max(np.abs(ux).max(), np.abs(uy).max()), 0.):
                dtmax = dtmax / CFL
                if u != 0 and D / u < dtmax:
                    dtmax = D / u
                dtmax *= CFL
                if dtmax > self.prev:
                    dtmax = (self.prev + 0.1 * dtmax) / 1.1
                self.prev = dtmax
        return dq, dtmax


class PeriodicNumpyStochasticModel(PeriodicNumpyModel):
    """the stochastic stage updates (float dts, a libc rand() field at every other stage) of NumpyStochasticModel"""
    generate_noise = NumpyStochasticModel.generate_noise
    advance = NumpyStochasticModel.advance
    step = NumpyStochasticModel.step

    def __init__(self, kw, psi, sigma, libc):
        super().__init__(kw, psi, stochastic=True)
        self.sigma, self.libc = sigma, libc
        self.corrector_step = 0
        self.noise = np.zeros_like(psi)


def _oracle(kw, psi, sigma=None):
    m = O.Model(O.make_params(**kw)); m.set_smoother("rb")
    m.set(O.PSI, psi)
    if sigma is not None:
        m.set(O.SSTOCH, sigma)
    m.set_const()
    return m


@pytest.mark.parametrize("N,nl,nsteps", [(32, 2, 4), (32, 3, 3)])
def test_periodic_timesteps_against_numpy_restatement(N, nl, nsteps):
    kw = base_kw(N, nl, sbc=-1.)
    psi = periodic_psi(N, nl)
    m = _oracle(kw, psi)
    ref = PeriodicNumpyModel(kw, psi)
    assert np.abs(ref.q - m.get(O.Q)).max() <= 1e-12 * np.abs(ref.q).max()
    for k in range(nsteps):
        dto, dtn = m.step(), ref.step()
        assert dto == pytest.approx(dtn, rel=1e-11), k
    assert m.L.orc_total_cycles(m.h) == ref.cycles
    for a, b in ((m.get(O.Q), ref.q), (m.get(O.PSI), ref.psi)):
        assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max()


def test_periodic_stochastic_timesteps_against_numpy_restatement():
    libc = C.CDLL(None)
    N, nl, nsteps = 32, 3, 3
    kw = base_kw(N, nl, sbc=-1., stochastic=1, tr_stoch=10., amp_stoch=1.)
    psi = periodic_psi(N, nl)
    sigma = 1e-3 * (1 + np.arange(nl)[:, None, None]) * np.ones((nl, N, N))
    m = _oracle(kw, psi, sigma)
    libc.srand(77)
    dto = [m.step() for _ in range(nsteps)]
    ref = PeriodicNumpyStochasticModel(kw, psi, sigma, libc)
    libc.srand(77)
    dtn = [ref.step() for _ in range(nsteps)]
    assert dto == pytest.approx(dtn, rel=1e-11)
    assert m.L.orc_total_cycles(m.h) == ref.cycles
    noise = m.get(O.NSTOCH)
    assert np.abs(noise - ref.noise).max() <= 1e-15 * np.abs(noise).max() and np.abs(noise).max() > 0
    for a, b in ((m.get(O.Q), ref.q), (m.get(O.PSI), ref.psi)):
        assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max()
    # the noise and the stochastic right-hand side really act: the deterministic periodic run differs
    det = _oracle(base_kw(N, nl, sbc=-1.), psi)
    for _ in range(nsteps):
        det.step()
    assert np.abs(det.get(O.Q) - m.get(O.Q)).max() > 1e-6 * np.abs(m.get(O.Q)).max()
