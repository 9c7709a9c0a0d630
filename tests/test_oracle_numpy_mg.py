"""The whole PV inversion -- poisson_layer (msqg/poisson_layer.h:263-306) -> [BASILISK] mg_solve / mg_cycle (in-tree copy
mspg/elliptic.h:43-99, :145-229) with relax_layer in red-black order and residual_layer -- restated a second time in
whole-array numpy and run beside the C oracle: same number of cycles, same nrelax history, same residual norms and the
same stream function to round-off, for a cold start (several cycles, nrelax adapts) and a warm start.  The red-black
ordering is what makes this possible: a half-sweep is one vectorised update of all cells of a colour.  What this pins
beyond the sweep itself (tests/test_oracle_rb.py): restriction of the residual AND of the stretching on every call,
minlevel = 1, zero initial guess on the coarsest level, bilinear prolongation with homogeneous ghosts, nrelax sweeps
per level, the correction, NITERMIN = 1, the unscaled max-norm test against 1e-3 (qg.h:159) and the nrelax
adaptation.  (CPU test, no GPU.)"""
import numpy as np
import pytest

from common import base_kw, synth_psi
from oracle import oracle as O
from test_oracle_numpy_rhs import lap, pad, sh, stretch
from test_oracle_rb import _numpy_rb_sweeps


def restrict(f):
    return 0.25 * (f[:, 0::2, 0::2] + f[:, 1::2, 0::2] + f[:, 0::2, 1::2] + f[:, 1::2, 1::2])


def prolong(c, bc=-1):
    nl, nc = c.shape[0], c.shape[1]
    out = np.zeros((nl, 2 * nc, 2 * nc))
    for l in range(nl):
        C = pad(c[l], bc)
        for py in (0, 1):
            for px in (0, 1):
                cx, cy = (1 if px else -1), (1 if py else -1)
                out[l, py::2, px::2] = (9. * sh(C, 0, 0) + 3. * (sh(C, cx, 0) + sh(C, 0, cy)) + sh(C, cx, cy)) / 16.
    return out


def residual(a, b, s, idh0, idh1, D, bc=-1):
    A = [pad(a[l], bc) for l in range(a.shape[0])]
    r = b - np.array([lap(A[l], D) for l in range(a.shape[0])]) - stretch(a, list(s), idh0, idh1)
    return r, float(np.abs(r).max())


def numpy_solve(a, b, s_fine, dh, L0, tol=1e-3, bc=-1, schedule=None):
    """bc = -1: closed basin (dirichlet(0)); bc = 0: doubly periodic (sbc = -1, qg.h:842-846).
    schedule: exactly len(schedule) cycles, cycle k with schedule[k] sweeps per level, no tolerance stop and no nrelax
    adaptation (orc_test_cycles).  stats["resas"] holds the residual after every cycle."""
    nl, N = a.shape[0], a.shape[1]
    depth = int(np.log2(N))
    dhc = 0.5 * (dh[:-1] + dh[1:])
    idh0 = np.zeros(nl); idh1 = np.zeros(nl)
    idh1[:-1] = 1. / (dhc * dh[:-1]); idh0[1:] = 1. / (dhc * dh[1:])
    s_lev = {depth: s_fine}
    for l in range(depth - 1, 0, -1):            # restriction(strl), poisson_layer.h:284
        s_lev[l] = restrict(s_lev[l + 1])
    a = a.copy()
    hist = []
    res, resb = residual(a, b, s_fine, idh0, idh1, L0 / N, bc)
    stats = dict(resb=resb, resa=resb, nrelax=4, i=0, resas=[])
    while (stats["i"] < len(schedule)) if schedule is not None else (stats["i"] < 100 and (stats["i"] < 1 or stats["resa"] > tol)):
        if schedule is not None:
            stats["nrelax"] = schedule[stats["i"]]
        # mg_cycle with minlevel = 1
        r_lev = {depth: res}
        for l in range(depth - 1, 0, -1):
            r_lev[l] = restrict(r_lev[l + 1])
        da = None
        for l in range(1, depth + 1):
            n = 1 << l
            da = np.zeros((nl, n, n)) if l == 1 else prolong(da, bc)
            da = _numpy_rb_sweeps(nl, n, L0, list(dh), s_lev[l], da, r_lev[l], stats["nrelax"], periodic=(bc == 0))
        a = a + da
        hist.append(stats["nrelax"])
        res, resa = residual(a, b, s_fine, idh0, idh1, L0 / N, bc)
        stats["resa"] = resa
        stats["resas"].append(resa)
        if schedule is None and resa > tol:
            if resb / resa < 1.2 and stats["nrelax"] < 100:
                stats["nrelax"] += 1
            elif resb / resa > 10 and stats["nrelax"] > 2:
                stats["nrelax"] -= 1
        resb = resa
        stats["i"] += 1
    return a, stats, hist


@pytest.mark.parametrize("N,nl,varRo", [(64, 2, 0), (64, 3, 0), (32, 4, 1), (64, 7, 0), (64, 12, 0), (32, 6, 1)])
def test_inversion_against_numpy_multigrid(N, nl, varRo):
    kw = base_kw(N, nl, varRo=varRo)
    m = O.Model(O.make_params(**kw)); m.set_smoother("rb")
    psi0 = synth_psi(N, nl)
    m.set(O.PSI, psi0); m.set_const()
    q = m.get(O.Q)
    strl = m.get(O.STR)[:nl - 1]
    dh = np.array(kw["dh"], dtype=float)
    for start in (np.zeros_like(psi0), psi0 * (1 + 1e-3)):      # cold start; warm start close to the solution
        m.set(O.PSI, start); m.invertq()
        so = m.mgstats()
        ref, st, hist = numpy_solve(start, q, strl, dh, kw["L0"])
        assert (so.i, so.nrelax) == (st["i"], st["nrelax"]), (so.i, so.nrelax, st, hist)
        assert so.resb == pytest.approx(st["resb"], rel=1e-10) and so.resa == pytest.approx(st["resa"], rel=1e-8)
        got = m.get(O.PSI)
        assert np.abs(got - ref).max() <= 1e-11 * np.abs(ref).max()
    assert so.i >= 1


@pytest.mark.parametrize("N,nl", [(32, 2), (64, 3), (64, 7), (64, 10), (64, 12)])
def test_periodic_inversion_against_numpy_multigrid(N, nl):
    """sbc = -1: the same solve with wrap-around ghost rings on every level (np.pad(..., mode="wrap") in the numpy
    version, boundary_level() in the oracle) -- relaxation across the seam, prolongation from the wrapped coarse ring,
    residual; down to the 2 x 2 level, where east and west neighbour are the same cell."""
    from common import periodic_psi
    kw = base_kw(N, nl, sbc=-1.)
    m = O.Model(O.make_params(**kw)); m.set_smoother("rb")
    psi0 = periodic_psi(N, nl)
    m.set(O.PSI, psi0); m.set_const()
    q = m.get(O.Q)
    D = kw["L0"] / N
    dh = np.array(kw["dh"], dtype=float)
    dhc = 0.5 * (dh[:-1] + dh[1:])
    idh0 = np.zeros(nl); idh1 = np.zeros(nl)
    idh1[:-1] = 1. / (dhc * dh[:-1]); idh0[1:] = 1. / (dhc * dh[1:])
    strl = m.get(O.STR)[:nl - 1]
    qn = np.array([lap(pad(psi0[l], 0), D) for l in range(nl)]) + stretch(psi0, list(strl), idh0, idh1)   # comp_q, periodic
    assert np.abs(qn - q).max() <= 1e-12 * np.abs(q).max()
    for start in (np.zeros_like(psi0), psi0 * (1 + 1e-3)):
        m.set(O.PSI, start); m.invertq()
        so = m.mgstats()
        ref, st, hist = numpy_solve(start, q, strl, dh, kw["L0"], bc=0)
        assert (so.i, so.nrelax) == (st["i"], st["nrelax"]), (so.i, so.nrelax, st, hist)
        assert so.resa == pytest.approx(st["resa"], rel=1e-8)
        got = m.get(O.PSI)
        assert np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max()


def test_reference_order_sweep_against_python_loops():
    """relax_layer in the REFERENCE order (msqg/poisson_layer.h:75-149: in place, [BASILISK] foreach = x outer, y inner),
    cell by cell in plain Python with a dense solve of each column's tridiagonal system (numpy.linalg.solve instead of
    the Thomas recurrence): the lexicographic path of the oracle -- the parity path of the CUDA library -- to round-off."""
    nl, level, L0, nsweeps = 3, 4, 80., 2
    n = 1 << level
    D = L0 / n
    rng = np.random.default_rng(33)
    dh = np.array([0.06, 0.14, 0.8])
    dhc = 0.5 * (dh[:-1] + dh[1:])
    idh0 = np.zeros(nl); idh1 = np.zeros(nl)
    idh1[:-1] = 1. / (dhc * dh[:-1]); idh0[1:] = 1. / (dhc * dh[1:])
    s = np.abs(rng.standard_normal((nl - 1, n, n))) * 5 + 8
    a = rng.standard_normal((nl, n, n)); b = rng.standard_normal((nl, n, n))
    got = a.copy()
    O.lib().orc_test_relax(nl, level, L0, dh, np.ascontiguousarray(s), got, b, nsweeps, 1, 1)
    g = np.zeros((nl, n + 2, n + 2))                 # [l][y][x] with one ghost ring
    g[:, 1:-1, 1:-1] = a

    def ghosts():
        g[:, 1:-1, 0] = -g[:, 1:-1, 1]; g[:, 1:-1, -1] = -g[:, 1:-1, -2]
        g[:, 0, :] = -g[:, 1, :]; g[:, -1, :] = -g[:, -2, :]

    ghosts()
    for _ in range(nsweeps):
        for i in range(n):                           # x outer
            for j in range(n):                       # y inner
                A = np.zeros((nl, nl)); r = np.zeros(nl)
                for l in range(nl):
                    lo = s[l - 1, j, i] * idh0[l] if l > 0 else 0.
                    up = s[l, j, i] * idh1[l] if l < nl - 1 else 0.
                    # -Delta^2 (laplacian(a) + Gamma(a) = b) solved for the column, neighbours taken as they are
                    A[l, l] = 4. + D * D * (lo + up)
                    if l > 0:
                        A[l, l - 1] = -D * D * lo
                    if l < nl - 1:
                        A[l, l + 1] = -D * D * up
                    r[l] = -D * D * b[l, j, i] + g[l, j + 1, i + 2] + g[l, j + 1, i] + g[l, j + 2, i + 1] + g[l, j, i + 1]
                g[:, j + 1, i + 1] = np.linalg.solve(A, r)
        ghosts()                                     # boundary_level after the sweep: ghosts keep the pre-sweep values during it
    assert np.abs(g[:, 1:-1, 1:-1] - got).max() <= 1e-11 * np.abs(got).max()
