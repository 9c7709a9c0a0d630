"""Multigrid correction folded into the last streaming red-black relax pass (k_relax_rb<..., FOLD = true>).

The last pass on the finest level adds da to the unknown with its ghost ring instead of storing da (no k_correct).
MSQG_RB_FOLD=0 restores the separate launch.  Both settings must give the oracle's bits, the same multigrid statistics
and cycle counts; folding must launch fewer kernels wherever it applies (nl <= 8 and the scalar modal solves, finest
level above the one-window kernel)."""
import numpy as np
import pytest

from common import make_pair

pytestmark = pytest.mark.gpu


def _fr_field(N, nl):
    y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
    fr = np.zeros((nl, N, N))
    for l in range(nl - 1):
        fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y))
    return fr


def _run(N, nl, over, frfield, cold, nsteps, with_oracle):
    """cold-start invertq (nrelax adapts, multi-pass splits) then nsteps steps (recorded cycle graphs replayed)"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, psi = make_pair(N, nl, smoother="rb", **over)
    models = [(mg, G)] + ([(mo, O)] if with_oracle else [])
    if frfield:
        for m, M in models:
            m.set(M.FR, _fr_field(N, nl))
    for m, _ in models:
        m.set_const()
    modes = range(nl) if over.get("mode_pv_invert") else [-1]
    out = []
    for m, M in models:
        stats = []
        if cold:
            m.set(M.PSI, np.zeros_like(psi))
            m.invertq()
            stats = [tuple((s.i, s.nrelax, s.resb, s.resa)) for s in (m.mgstats(k) for k in modes)]
            m.set(M.PSI, psi)
        dts = [m.step() for _ in range(nsteps)]
        cycles = m.total_cycles if M is G else m.L.orc_total_cycles(m.h)
        out.append(dict(psi=m.get(M.PSI), q=m.get(M.Q), stats=stats, dts=dts, cycles=cycles,
                        launches=m.launches if M is G else None))
    mg.close()
    return out


CASES = [
    # streaming kernel on every level (MSQG_RB_TILE=0): NSMAX 4 (nl 2-4), 2 (nl 5, 8: two passes, the second one
    # corrects) and 1 (nl 9, 12: no fold instance)
    (128, 2, {}, 0, "0"), (128, 3, {}, 0, "0"), (128, 4, {}, 0, "0"), (128, 5, {}, 0, "0"), (128, 8, {}, 0, "0"),
    (128, 9, {}, 0, "0"), (128, 12, {}, 0, "0"),
    (128, 3, dict(mode_pv_invert=1), 0, "0"),               # scalar modal solves (NL = 1 instance)
    (128, 3, dict(varRo=1), 0, "0"),                        # per-row coefficient tables
    (128, 4, {}, 1, "0"),                                   # Fr(x, y): per-cell coefficient tables
    (128, 3, dict(mode_pv_invert=1, varRo=1), 1, "0"),      # per-cell modal tables
]


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("N,nl,over,frfield,tile", CASES)
def test_fold_equals_separate_launches_and_oracle(gpu, N, nl, over, frfield, tile, graph, monkeypatch):
    from oracle import oracle as O
    if over.get("mode_pv_invert") and O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")
    if graph == "0" and (nl > 4 or over or frfield):
        pytest.skip("eager launches (MSQG_GRAPH=0) on the layer-coupled nl <= 4 cases only")
    monkeypatch.setenv("MSQG_RB_TILE", tile)
    monkeypatch.setenv("MSQG_GRAPH", graph)
    res = {}
    for fold in ("1", "0"):
        monkeypatch.setenv("MSQG_RB_FOLD", fold)
        res[fold] = _run(N, nl, over, frfield, cold=True, nsteps=4, with_oracle=fold == "1")
    on, off, orc = res["1"][0], res["0"][0], res["1"][1]
    for r in (off, orc):
        assert np.array_equal(on["psi"], r["psi"]) and np.array_equal(on["q"], r["q"])
        assert on["stats"] == r["stats"] and on["dts"] == r["dts"] and on["cycles"] == r["cycles"]
    print("nl %d: nrelax after the cold start %s, launches fold on / off %d / %d"
          % (nl, [s[1] for s in on["stats"]], on["launches"], off["launches"]))
    if nl <= 8:
        assert on["launches"] < off["launches"]
    else:
        assert on["launches"] == off["launches"]   # nl > 8: the single-stage instances keep k_correct


def test_fold_above_tiled_levels(gpu, monkeypatch):
    """default tile limit: the 1024^2 finest level streams above levels of the one-window kernel, and its last pass
    corrects psi"""
    res = {}
    for fold in ("1", "0"):
        monkeypatch.setenv("MSQG_RB_FOLD", fold)
        res[fold] = _run(1024, 4, {}, 0, cold=False, nsteps=2, with_oracle=fold == "1")
    on, off, orc = res["1"][0], res["0"][0], res["1"][1]
    for r in (off, orc):
        assert np.array_equal(on["psi"], r["psi"]) and np.array_equal(on["q"], r["q"])
        assert on["dts"] == r["dts"] and on["cycles"] == r["cycles"]
    assert on["launches"] < off["launches"]
