"""The residual pass of the multigrid solve with the restriction pyramid it writes (k_residual_pyr), bit for bit
against the oracle.

On one undecomposed, non-periodic grid the residual kernel also leaves res restricted down to level max(1, D - 5), so
that a cycle restricts only the levels below that.  Every level it writes must equal the oracle's residual followed by
repeated restriction, and the max-norm must be the oracle's.  Covered: the layer-coupled problem at several nl with
uniform stretching (per-layer constants) and per-cell stretching (read from the field), the scalar Helmholtz problem
of one vertical mode with uniform and varying lambda, grids from smaller than one 32x32 tile up to 1024^2, and inputs
with exact zeros."""
import ctypes as C

import numpy as np
import pytest

from common import base_kw, synth_psi

pytestmark = pytest.mark.gpu


def _fr_field(N, nl):
    y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
    fr = np.zeros((nl, N, N))
    for l in range(nl - 1):
        fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y))
    return fr


def _inputs(nf, N, seed, zeros):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((nf, N, N))
    b = rng.standard_normal((nf, N, N))
    if zeros:  # whole blocks of exact zeros (so that some quads restrict four zero children), and scattered ones
        for f in (a, b):
            f[:, : N // 2, : N // 2] = 0.0
            f[rng.random(f.shape) < 0.2] = 0.0
        b[:, N // 2:, : N // 4] = -0.0
    return a, b


def _run(gpu, nl, N, field, modal, zeros=False):
    from oracle import oracle as O
    from msom_b200 import capi as G
    over = dict(mode_pv_invert=1, varRo=int(field)) if modal else {}
    kw = base_kw(N, nl, **over)
    m = G.Model(G.make_params(**kw), gpu)
    m.set(G.PSI, synth_psi(N, nl))
    if field and not modal:
        m.set(G.FR, _fr_field(N, nl))
    m.set_const()
    mode = nl - 1 if modal else -1
    nf = 1 if modal else nl
    D = int(np.log2(N))
    a, b = _inputs(nf, N, 17 * N + nl, zeros)

    out = np.zeros(nf * sum(4 ** l for l in range(D + 1)))
    mx, bottom = C.c_double(), C.c_int()
    G.check(G.lib().msqg_test_residual_levels(m.h, mode, a, b, out, C.byref(mx), C.byref(bottom)))
    assert bottom.value == max(1, D - 5)

    r_ref = np.zeros_like(a)
    if modal:
        lam = np.ascontiguousarray(m.get(G.IBU)[mode:mode + 1])
        assert field or np.all(lam == lam.flat[0])
        assert not field or not np.all(lam == lam.flat[0])
        mx_ref = O.lib().orc_test_residual_scalar(D, kw["L0"], lam, a, b, r_ref)
    else:
        s = np.ascontiguousarray(m.get(G.STR)[: nl - 1])
        assert all(np.all(s[l] == s[l].flat[0]) != field for l in range(nl - 1))
        mx_ref = O.lib().orc_test_residual(nl, D, kw["L0"], np.array(kw["dh"], dtype=np.float64), s, a, b, r_ref)
    m.close()

    off, ref = 0, r_ref
    for lev in range(D, bottom.value - 1, -1):
        n = 1 << lev
        got = out[off: off + nf * n * n].reshape(nf, n, n)
        off += nf * n * n
        if lev < D:
            coarse = np.zeros((nf, n, n))
            O.lib().orc_test_restrict(nf, lev + 1, np.ascontiguousarray(ref), coarse)
            ref = coarse
        assert np.array_equal(got, ref), (lev, float(np.abs(got - ref).max()))
        assert np.array_equal(np.signbit(got), np.signbit(ref)), lev
    assert mx.value == mx_ref


CASES = (
    # layer-coupled: every nl at 64^2, uniform and per-cell stretching
    [(nl, 64, field) for nl in (2, 4, 5, 8, 12) for field in (False, True)]
    # grids of one tile, of less than one tile, and larger ones
    + [(2, 16, False), (4, 16, True), (4, 32, False), (12, 32, True), (5, 256, False), (8, 256, True), (12, 256, False),
       (4, 1024, False), (2, 1024, True)]
)


@pytest.mark.parametrize("nl,N,field", CASES)
def test_residual_pyramid_layers(gpu, nl, N, field):
    _run(gpu, nl, N, field, modal=False)


@pytest.mark.parametrize("N,field", [(16, False), (32, True), (64, False), (64, True), (256, True), (1024, False)])
def test_residual_pyramid_scalar_mode(gpu, N, field):
    _run(gpu, 3, N, field, modal=True)


@pytest.mark.parametrize("nl,N,modal", [(4, 128, False), (3, 64, True)])
def test_residual_pyramid_exact_zeros(gpu, nl, N, modal):
    _run(gpu, nl, N, True, modal, zeros=True)
