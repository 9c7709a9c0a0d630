"""Throughput mode: red-black ordering of the relaxation sweep (msqg_set_smoother(m, 1), rb_kernels.cuh).

The cell update is the reference's (msqg/poisson_layer.h:80-146); only the traversal differs, which the reference
itself documents as implementation dependent (poisson_layer.h:55-65).  The CUDA path is checked bit for bit against
the oracle running the same ordering (orc_set_smoother), with equal multigrid cycle counts; against the
reference-order (lexicographic) solution it agrees to the solver tolerance."""
import numpy as np
import pytest

from common import DH, FR, base_kw, make_pair, rel_l2, synth_psi

pytestmark = pytest.mark.gpu


def _model(gpu, N, nl, **over):
    from msom_b200 import capi as G
    m = G.Model(G.make_params(**base_kw(N, nl, **over)), gpu)
    m.set_smoother("rb")
    m.set(G.PSI, synth_psi(N, nl))
    m.set_const()
    return m


def _level_s(N, nl, level, kw):
    n = 1 << level
    s = np.zeros((nl - 1, n, n))
    for l in range(nl - 1):
        v = (kw["Fr"][l] / kw["Rom"]) ** 2
        for _ in range(int(np.log2(N)) - level):
            v = (((0.0 + v) + v) + v + v) / 4
        s[l] = v
    return s


@pytest.mark.parametrize("nl,level,nsweeps", [(2, 3, 1), (2, 5, 4), (3, 6, 4), (4, 7, 4), (4, 6, 3), (4, 5, 2), (4, 8, 1),
                                               (3, 7, 7), (2, 6, 13), (10, 5, 4), (4, 1, 4), (4, 2, 5), (2, 8, 4),
                                               (4, 9, 4), (6, 7, 3), (12, 6, 2), (4, 10, 6),
                                               # every layer count of the streaming kernel: 2 fused sweeps per pass for nl
                                               # 5-8 (odd nl: uneven plane split), 1 for nl 9-12; several strips from level 7
                                               (5, 7, 5), (7, 8, 3), (8, 7, 4), (9, 8, 3), (11, 7, 2), (11, 9, 1)])
# wxmin is not read any more (it sized a window variant that was removed); it stays so that the test ids stay the same
@pytest.mark.parametrize("reuse,tile,wxmin", [(1, 0, 1024), (0, 0, 1024), (1, 512, 1024)])
def test_relax_rb_matches_oracle(gpu, nl, level, nsweeps, reuse, tile, wxmin, monkeypatch):
    """one level, nsweeps red-black sweeps: strips, row chunks, window halos and multi-pass splits all exercised, with the
    streaming kernel (MSQG_RB_TILE=0 forces it on every size) and with the one-window-per-CTA kernel of the small levels"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    if reuse == 0 and level > 8:
        pytest.skip("register-reuse A/B on the smaller levels only")
    monkeypatch.setenv("MSQG_RB_REUSE", str(reuse))
    monkeypatch.setenv("MSQG_RB_TILE", str(tile))
    N = max(1 << level, 32)
    m = _model(gpu, N, nl)
    n = 1 << level
    rng = np.random.default_rng(100 + level)
    a = rng.standard_normal((nl, n, n))
    b = rng.standard_normal((nl, n, n))
    kw = base_kw(N, nl)
    s = _level_s(N, nl, level, kw)
    a_ref = a.copy()
    dh = np.array(kw["dh"], dtype=np.float64)
    O.lib().orc_test_relax_rb(nl, level, kw["L0"], dh, s, a_ref, b, nsweeps)
    a_gpu = a.copy()
    G.check(G.lib().msqg_test_relax(m.h, level, a_gpu, b, nsweeps))
    assert np.array_equal(a_gpu, a_ref), np.abs(a_gpu - a_ref).max()


@pytest.mark.parametrize("level,nsweeps,lam", [(4, 4, 0.0), (6, 4, -3.7), (7, 2, -50.0), (5, 8, -0.3), (9, 5, -1.0)])
@pytest.mark.parametrize("tile", [0, 512])
def test_relax_rb_scalar_matches_oracle(gpu, level, nsweeps, lam, tile, monkeypatch):
    from oracle import oracle as O
    from msom_b200 import capi as G
    monkeypatch.setenv("MSQG_RB_TILE", str(tile))
    N = max(1 << level, 32)
    m = _model(gpu, N, 2)
    n = 1 << level
    rng = np.random.default_rng(5 + level)
    a = rng.standard_normal((1, n, n)); b = rng.standard_normal((1, n, n))
    a_ref = a.copy()
    O.lib().orc_test_relax_scalar_rb(level, 80., np.full((1, n, n), lam), a_ref, b, nsweeps)
    a_gpu = a.copy()
    G.check(G.lib().msqg_test_relax_scalar(m.h, level, lam, a_gpu, b, nsweeps))
    assert np.array_equal(a_gpu, a_ref), np.abs(a_gpu - a_ref).max()


NL_HIGH = range(5, 13)   # layer counts above the one-window relax kernel: 2 (nl <= 8) or 1 fused sweeps per pass


@pytest.mark.parametrize("N,nl", [(64, 2), (256, 2), (128, 3), (128, 4), (64, 10)] + [(256, nl) for nl in NL_HIGH])
def test_invertq_rb(gpu, N, nl):
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, psi = make_pair(N, nl, smoother="rb")
    mo.set_const(); mg.set_const()
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()
    so, sg = mo.mgstats(), mg.mgstats()
    assert (sg.i, sg.nrelax) == (so.i, so.nrelax)
    assert sg.resb == so.resb and sg.resa == so.resa
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))


@pytest.mark.parametrize("N,nl,nsteps", [(256, 2, 1), (256, 2, 100), (128, 3, 20), (128, 4, 20), (512, 4, 3)]
                         + [(256, nl, 3) for nl in NL_HIGH])
def test_steps_rb(gpu, N, nl, nsteps):
    """BASELINE config 1 (256^2 x 2) in throughput mode: 1 and 100 steps, bit-exact against the oracle with the same
    ordering, equal multigrid cycle counts"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(N, nl, smoother="rb")
    mo.set_const(); mg.set_const()
    for _ in range(nsteps):
        dto = mo.step()
        dtg = mg.step()
        assert dtg == dto
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    for fg, fo in ((G.PSI, O.PSI), (G.Q, O.Q)):
        a, b = mg.get(fg), mo.get(fo)
        assert np.array_equal(a, b), rel_l2(a, b)


def test_rb_agrees_with_reference_order_to_solver_tolerance(gpu):
    """rb and lex iterates solve the same elliptic problem to the same tolerance (1e-3 on max|res|, qg.h:159): after 10
    steps the states differ by O(tolerance), far above round-off and far below the signal; cycle counts are recorded"""
    from msom_b200 import capi as G
    out = {}
    for sm in ("lex", "rb"):
        m = G.Model(G.make_params(**base_kw(256, 4)), gpu)
        m.set_smoother(sm)
        m.set(G.PSI, synth_psi(256, 4))
        m.set_const()
        for _ in range(10):
            m.step()
        out[sm] = (m.get(G.PSI), m.get(G.Q), m.total_cycles, m.mgstats().resa)
        m.close()
    dpsi, dq = rel_l2(out["rb"][0], out["lex"][0]), rel_l2(out["rb"][1], out["lex"][1])
    print("cycles lex/rb: %d/%d, rel L2 difference psi %.3e q %.3e" % (out["lex"][2], out["rb"][2], dpsi, dq))
    assert out["rb"][3] <= 1e-3 and out["lex"][3] <= 1e-3       # both converged to the reference's tolerance
    assert 0 < dpsi < 5e-3 and 0 < dq < 5e-3
    assert abs(out["rb"][2] - out["lex"][2]) <= out["lex"][2] // 2


def test_varro_rb(gpu):
    """stretching that depends on y (varRo > 0): per-row coefficient tables in the rb kernel"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(128, 3, smoother="rb", varRo=1)
    mo.set_const(); mg.set_const()
    for _ in range(3):
        assert mg.step() == mo.step()
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))


def test_modal_rb(gpu):
    """vertical-mode inversion (MODE_PV_INVERT 1): scalar Helmholtz solves with the rb ordering"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(128, 3, smoother="rb", mode_pv_invert=1)
    mo.set_const(); mg.set_const()
    for _ in range(3):
        assert mg.step() == mo.step()
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))


@pytest.mark.parametrize("N,nl,over", [(256, 4, {}), (128, 3, {"mode_pv_invert": 1}), (64, 10, {}), (16, 2, {}),
                                       (128, 9, {}), (128, 12, {})])   # coarse kernel up to 32^2 at nl = 9, up to 16^2 at nl = 12
def test_fused_coarse_levels_equal_level_by_level(gpu, N, nl, over, monkeypatch):
    """k_coarse_rb (levels up to 32^2 in one launch, restrictions and prolongations included) against the
    level-by-level kernels (MSQG_RB_COARSE=0) and against the oracle: same bits, same cycle counts"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    res = []
    for flag in ("1", "0"):
        monkeypatch.setenv("MSQG_RB_COARSE", flag)
        mo, mg, psi = make_pair(N, nl, smoother="rb", **over)
        mo.set_const(); mg.set_const()
        z = np.zeros_like(psi)
        mg.set(G.PSI, z)
        mg.invertq()
        for _ in range(3):
            mg.step()
        res.append((mg.get(G.PSI), mg.get(G.Q), mg.total_cycles, mg.launches))
        if flag == "1":
            mo.set(O.PSI, z); mo.invertq()
            for _ in range(3):
                mo.step()
            assert np.array_equal(res[0][0], mo.get(O.PSI)) and np.array_equal(res[0][1], mo.get(O.Q))
            assert res[0][2] == mo.L.orc_total_cycles(mo.h)
        mg.close()
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    assert res[0][2] == res[1][2]
    assert res[0][3] < res[1][3]      # fewer launches


def test_rb_against_committed_golden_fixture(gpu):
    """the CUDA path against the committed fixture of the oracle (regression fixture, tests/golden/make_golden.py)"""
    import os
    from msom_b200 import capi as G
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_rb_32x2_3steps.npz"))
    m = _model(gpu, 32, 2)
    dts = [m.step() for _ in range(3)]
    assert np.array_equal(np.array(dts), g["dts"])
    assert np.array_equal(m.get(G.PSI), g["psi"]) and np.array_equal(m.get(G.Q), g["q"])


@pytest.mark.parametrize("tables", ["1", "0"])
@pytest.mark.parametrize("N,nl,over,frfield", [(256, 3, dict(varRo=1), 0), (128, 4, {}, 1), (128, 3, dict(mode_pv_invert=1, varRo=1), 1),
                                                 (64, 2, dict(mode_pv_invert=1), 1)])
def test_coefficient_tables_in_the_small_level_kernels(gpu, N, nl, over, frfield, tables, monkeypatch):
    """Horizontally varying stretching (varRo, Fr(x, y)) and varying vertical modes: the one-window-per-CTA kernel and the
    single-CTA coarse kernel read the same per-row / per-cell Thomas coefficient tables as the streaming kernel
    (MSQG_RB_COARSE_TABLES=0 sends every level through the streaming kernel, the first implementation): both give the
    bits of the oracle, with equal cycle counts."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    if over.get("mode_pv_invert") and O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")
    monkeypatch.setenv("MSQG_RB_COARSE_TABLES", tables)
    mo, mg, psi = make_pair(N, nl, smoother="rb", **over)
    if frfield:
        y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
        fr = np.zeros_like(psi)
        for l in range(nl - 1):
            fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y))
        mo.set(O.FR, fr); mg.set(G.FR, fr)
    mo.set_const(); mg.set_const()
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()                      # cold start: several cycles, nrelax adapts
    for mode in ([-1] if not over.get("mode_pv_invert") else range(nl)):
        so, sg = mo.mgstats(mode), mg.mgstats(mode)
        assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa), mode
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    mo.set(O.PSI, psi); mg.set(G.PSI, psi)
    for _ in range(4):                              # enough steps for the recorded cycle graphs to be replayed
        assert mg.step() == mo.step()
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI)) and np.array_equal(mg.get(G.Q), mo.get(O.Q))


def test_round2_variants_against_committed_golden_fixtures(gpu):
    """periodic domain (red-black), ENERGY_CONSERV (reference order) and per-column vertical modes against the committed
    fixtures of the oracle (tests/golden/make_golden.py; regression fixtures)"""
    import os
    from common import periodic_psi
    from oracle import oracle as O
    from msom_b200 import capi as G
    gdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    g = np.load(os.path.join(gdir, "oracle_rb_periodic_32x3_3steps.npz"))
    m = G.Model(G.make_params(**base_kw(32, 3, sbc=-1.)), gpu)
    m.set(G.PSI, periodic_psi(32, 3)); m.set_const()
    dts = [m.step() for _ in range(3)]
    assert np.array_equal(np.array(dts), g["dts"])
    assert np.array_equal(m.get(G.PSI), g["psi"]) and np.array_equal(m.get(G.Q), g["q"])
    g = np.load(os.path.join(gdir, "oracle_econs_32x2_3steps.npz"))
    m = G.Model(G.make_params(**base_kw(32, 2)), gpu)
    m.set_energy_conserv(1)
    m.set(G.PSI, synth_psi(32, 2)); m.set_const()
    dts = [m.step() for _ in range(3)]
    assert np.array_equal(np.array(dts), g["dts"])
    assert np.array_equal(m.get(G.PSI), g["psi"]) and np.array_equal(m.get(G.Q), g["q"])
    if O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")
    g = np.load(os.path.join(gdir, "oracle_32x3_modal_varRo_2steps.npz"))
    m = G.Model(G.make_params(**base_kw(32, 3, mode_pv_invert=1, varRo=1)), gpu)
    m.set(G.PSI, synth_psi(32, 3)); m.set_const()
    dts = [m.step() for _ in range(2)]
    assert np.array_equal(np.array(dts), g["dts"])
    assert rel_l2(m.get(G.PSI), g["psi"]) < 1e-11   # LAPACK builds may differ in the last bits
