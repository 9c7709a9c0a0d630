"""Multigrid cycles at every sweep count the adaptive solve can reach (nrelax 2..100), against the oracle.

mg_solve starts at nrelax = 4 and moves it by one per cycle (up when a cycle gains less than 1.2x, down when it gains more
than 10x).  A solve that converges in a few cycles only ever runs 3 and 4; one whose tolerance is below the round-off
floor of a large q climbs to 80 and more.  Many paths depend on nrelax: the red-black pass split and the fold of the
correction into the last pass, the da/da2 parity that keys the cycle graphs, the K = 4 launches of the reference-order
sweep, the run-time loop of k_coarse_rb, and the exchange chunks of at most 7 sweeps of a red-black tile group.

msqg_test_cycles runs the production solve loop with a fixed schedule (cycle k with nrelax[k] sweeps, no tolerance stop):
each value repeats six times, so every (nrelax, da parity) graph key is run eagerly, recorded and replayed.  The residual
after every cycle and the final unknown must be the oracle's bits (orc_test_cycles), and a group must give the bits of
the undecomposed model.  The last tests run stalled solves end to end through invertq."""
import numpy as np
import pytest

from common import base_kw, periodic_psi, synth_psi

pytestmark = pytest.mark.gpu

# each value six times in a row: a level's da parity can flip every cycle, so each (nrelax, parity) key gets its eager
# run, its recording and a replay
SCHED = [n for n in (2, 3, 4, 5, 6, 7, 8, 9, 13, 16, 17) for _ in range(6)] + [100]
# tile groups: 7 and 14 end a chunk of 7 exactly, 8, 15, 16 and 22 need a second or third exchange per level
GROUP_SCHED = [n for n in (2, 3, 4, 5, 6, 7, 8, 9, 13, 14, 15, 16, 17, 22) for _ in range(6)] + [100]
SHORT_SCHED = [n for n in (2, 5, 7, 8, 14, 15, 16, 22) for _ in range(3)] + [100]


def _fr_field(N, nl):
    y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
    fr = np.zeros((nl, N, N))
    for l in range(nl - 1):
        fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y))
    return fr


def _need_lapack(over):
    from oracle import oracle as O
    if over.get("mode_pv_invert") and O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")


def _inputs(N, nl, over):
    """psi for set_const, the start of the unknown, and (modal problems) the right-hand side of every mode"""
    psi = periodic_psi(N, nl) if over.get("sbc") == -1. else synth_psi(N, nl)
    return psi, np.zeros_like(psi), (0.01 * synth_psi(N, nl, seed=77) if over.get("mode_pv_invert") else None)


def _prepare(m, M, N, nl, over, frfield, setf):
    """set_const from psi, then the start of the cycles: unknown = 0 (PSI, or every plane of PM with QM as rhs)"""
    psi, start, qm = _inputs(N, nl, over)
    setf(M.PSI, psi)
    if frfield:
        setf(M.FR, _fr_field(N, nl))
    m.set_const()
    if qm is None:
        setf(M.PSI, start)
    else:
        setf(M.PM, start); setf(M.QM, qm)
    return M.PSI if qm is None else M.PM


_ORACLE = {}


def oracle_cycles(N, nl, over, sched, mode=-1, smoother="rb", frfield=0, decomp=None):
    """(resa per cycle, final unknown) of orc_test_cycles, computed once per configuration for the whole module"""
    from oracle import oracle as O
    key = (N, nl, tuple(sorted(over.items())), tuple(sched), mode, smoother, frfield, decomp)
    if key not in _ORACLE:
        mo = O.Model(O.make_params(**base_kw(N, nl, **over))); mo.set_smoother(smoother)
        if decomp:
            mo.L.orc_set_decomp(mo.h, *decomp)
        fid = _prepare(mo, O, N, nl, over, frfield, mo.set)
        resa = mo.test_cycles(sched, mode)
        _ORACLE[key] = (resa, mo.get(fid))
        mo.close()
    return _ORACLE[key]


def gpu_cycles(gpu, N, nl, over, sched, mode=-1, smoother="rb", frfield=0):
    from msom_b200 import capi as G
    m = G.Model(G.make_params(**base_kw(N, nl, **over)), gpu); m.set_smoother(smoother)
    fid = _prepare(m, G, N, nl, over, frfield, m.set)
    l0 = m.launches
    resa = m.test_cycles(sched, mode)
    out = dict(resa=resa, a=m.get(fid), launches=m.launches - l0)
    m.close()
    return out


def group_cycles(gpu, N, nl, over, sched, px, py, agg_n, mode=-1, smoother="rb"):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    g = Group(G.make_params(**base_kw(N, nl, **over)), px, py, agg_n, gpu, smoother=smoother)
    fid = _prepare(g, G, N, nl, over, 0, g.set_global)
    resa = g.test_cycles(sched, mode)
    out = dict(resa=resa, a=g.get_global(fid), transport=g.transport)
    if smoother == "rb":   # the exchanges of one cycle at 7 and at 8 sweeps (eager: first use of each key)
        x = [g.exchanges]
        for n in (7, 8):
            g.test_cycles([n], mode)
            x.append(g.exchanges)
        out["xchg"] = (x[1] - x[0], x[2] - x[1])
    g.close()
    return out


def _same(got, ref):
    resa, a = ref
    assert np.array_equal(got["resa"], resa), "resa differs after cycles %s" % list(np.nonzero(got["resa"] != resa)[0])
    d = np.abs(got["a"] - a)
    assert np.array_equal(got["a"], a), "unknown: max |difference| %.3e at %d cells" % (d.max(), int((d > 0).sum()))


# ------------------------------------------------------------------ single grid, red-black
@pytest.mark.parametrize("nl", [2, 3, 4, 5, 8, 9, 12])
def test_streaming_kernel_fold_on_and_off(gpu, nl, monkeypatch):
    """MSQG_RB_TILE=0: k_relax_rb on every level; NSMAX 4 (nl <= 4: several passes from nrelax 5 on, the fold in the last
    one), 2 (nl 5-8) and 1 (nl 9-12, no folded instance)"""
    monkeypatch.setenv("MSQG_RB_TILE", "0")
    ref = oracle_cycles(128, nl, {}, SCHED)
    runs = {}
    for fold in ("1", "0"):
        monkeypatch.setenv("MSQG_RB_FOLD", fold)
        runs[fold] = gpu_cycles(gpu, 128, nl, {}, SCHED)
        _same(runs[fold], ref)
    if nl <= 8:
        assert runs["1"]["launches"] < runs["0"]["launches"]
    else:
        assert runs["1"]["launches"] == runs["0"]["launches"]


@pytest.mark.parametrize("N,nl,sched", [(128, 2, SCHED), (128, 4, SCHED),
                                        # the fold on the streamed 1024^2 level above the levels of k_relax_rb_tile
                                        (1024, 4, [5] * 6 + [9] * 6 + [2] * 6)])
def test_default_tile_limit(gpu, N, nl, sched):
    """levels up to 512^2 through k_relax_rb_tile (several passes per level), the coarse levels in k_coarse_rb"""
    _same(gpu_cycles(gpu, N, nl, {}, sched), oracle_cycles(N, nl, {}, sched))


@pytest.mark.parametrize("env", [{"MSQG_GRAPH": "0"}, {"MSQG_RB_COARSE": "0"}, {"MSQG_GRAPH": "0", "MSQG_RB_TILE": "0"}],
                         ids=["eager", "level-by-level-coarse", "eager-streaming"])
def test_switches(gpu, env, monkeypatch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    _same(gpu_cycles(gpu, 128, 3, {}, SCHED), oracle_cycles(128, 3, {}, SCHED))


@pytest.mark.parametrize("nl,over,frfield,modes", [
    (3, dict(varRo=1), 0, [-1]),                    # per-row coefficient tables
    (4, {}, 1, [-1]),                               # Fr(x, y): per-cell tables
    (3, dict(mode_pv_invert=1), 0, [0, 2]),         # scalar modal solves, uniform modes
    (3, dict(mode_pv_invert=1, varRo=1), 0, [0, 2]),  # modes that vary with y: per-cell modal tables
], ids=["varRo", "frxy", "modal", "modal-varRo"])
def test_coefficient_tables(gpu, nl, over, frfield, modes):
    _need_lapack(over)
    for mode in modes:
        _same(gpu_cycles(gpu, 128, nl, over, SCHED, mode, frfield=frfield), oracle_cycles(128, nl, over, SCHED, mode, frfield=frfield))


# ------------------------------------------------------------------ single grid, reference order
@pytest.mark.parametrize("nl,cap", [(2, None), (4, None), (4, "3")], ids=["nl2", "nl4", "nl4-column-panels"])
def test_reference_order(gpu, nl, cap, monkeypatch):
    """the lexicographic sweep: more than 4 sweeps are consecutive launches of k_relax_ws<NL, 4>"""
    if cap:
        monkeypatch.setenv("MSQG_RELAX_CAP", cap)
    _same(gpu_cycles(gpu, 128, nl, {}, SCHED, smoother="lex"), oracle_cycles(128, nl, {}, SCHED, smoother="lex"))


# ------------------------------------------------------------------ tile groups
GROUPS = [
    # N, nl, px, py, agg_n, parameters, schedule
    (256, 4, 2, 2, 64, {}, GROUP_SCHED),
    (256, 3, 4, 2, 128, {}, GROUP_SCHED),
    (128, 2, 2, 2, 32, {}, GROUP_SCHED),         # 16-cell tiles: at 7 and 14 the last chunk exchanges a 15-cell halo
    (128, 7, 2, 2, 32, {}, GROUP_SCHED),         # 2 sweeps per tile pass
    (128, 12, 2, 1, 64, {}, SHORT_SCHED),        # 1 sweep per tile pass
    (256, 3, 2, 2, 64, dict(mode_pv_invert=1), SHORT_SCHED),
]


@pytest.mark.parametrize("p2p", [1, 0])
@pytest.mark.parametrize("N,nl,px,py,agg_n,over,sched", GROUPS)
def test_red_black_group(gpu, N, nl, px, py, agg_n, over, sched, p2p, monkeypatch):
    _need_lapack(over)
    monkeypatch.setenv("MSQG_P2P", str(p2p))
    for mode in ([0, nl - 1] if over.get("mode_pv_invert") else [-1]):
        ref = oracle_cycles(N, nl, over, sched, mode)
        got = group_cycles(gpu, N, nl, over, sched, px, py, agg_n, mode)
        assert got["transport"] == ("peer-memory" if p2p else "nccl")
        _same(got, ref)
        _same(gpu_cycles(gpu, N, nl, over, sched, mode), ref)
        x7, x8 = got["xchg"]
        assert x8 > x7, "a cycle at 8 sweeps must exchange da a second time on each distributed level (%d, %d)" % (x7, x8)


def test_reference_order_group(gpu):
    """block Gauss-Seidel on tiles, a one-cell halo exchanged after every sweep, against the oracle's emulation"""
    ref = oracle_cycles(128, 3, {}, SCHED, smoother="lex", decomp=(2, 2, 32))
    _same(group_cycles(gpu, 128, 3, {}, SCHED, 2, 2, 32, smoother="lex"), ref)


@pytest.mark.parametrize("N,nl,px,py", [(64, 3, 1, 1), (128, 4, 2, 1), (128, 3, 2, 2), (64, 10, 1, 1), (64, 10, 2, 2)])
def test_periodic(gpu, N, nl, px, py):
    """sbc = -1: the tile machinery with wrap-around halos (64^2 x 10 on 2 x 2: 16-cell tiles); the single-model handle
    dispatches to its 1 x 1 group"""
    over = dict(sbc=-1.)
    ref = oracle_cycles(N, nl, over, GROUP_SCHED)
    _same(group_cycles(gpu, N, nl, over, GROUP_SCHED, px, py, 0), ref)
    if px * py == 1:
        _same(gpu_cycles(gpu, N, nl, over, GROUP_SCHED), ref)


# ------------------------------------------------------------------ stalled solves, end to end
_STALLED = {}


def _stalled_oracle(N, nl, over, smoother):
    from oracle import oracle as O
    key = (N, nl, tuple(sorted(over.items())), smoother)
    if key not in _STALLED:
        mo = O.Model(O.make_params(**base_kw(N, nl, **over))); mo.set_smoother(smoother)
        _STALLED[key] = _stall(mo, O, N, nl, over, mo.set, mo.get)
    return _STALLED[key]


def _stall(m, M, N, nl, over, setf, getf):
    """q of psi * 1e13: the tolerance 1e-3 is below the residual's round-off floor, the solve runs 100 cycles"""
    psi, start, _ = _inputs(N, nl, over)
    setf(M.PSI, psi * 1e13); m.set_const()
    setf(M.PSI, start); m.invertq()
    modes = range(nl) if over.get("mode_pv_invert") else [-1]
    return [tuple((s.i, s.nrelax, s.resb, s.resa)) for s in (m.mgstats(k) for k in modes)], getf(M.PSI)


@pytest.mark.parametrize("N,nl,over,smoother,env,group", [
    (64, 4, {}, "rb", {}, None),
    (64, 4, {}, "rb", {"MSQG_RB_TILE": "0"}, None),
    (64, 4, {}, "lex", {}, None),
    (128, 3, {}, "rb", {}, (2, 2, 32)),
    (64, 3, dict(sbc=-1.), "rb", {}, None),
    (128, 3, dict(mode_pv_invert=1), "rb", {}, None),   # at 64^2 x 3 the modes still converge (nrelax <= 10)
], ids=["rb", "rb-streaming", "lex", "rb-group", "periodic", "modal"])
def test_stalled_solve(gpu, N, nl, over, smoother, env, group, monkeypatch):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    _need_lapack(over)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    stats, psi = _stalled_oracle(N, nl, over, smoother)
    p = G.make_params(**base_kw(N, nl, **over))
    if group:
        m = Group(p, *group, gpu, smoother=smoother)
        got = _stall(m, G, N, nl, over, m.set_global, m.get_global)
    else:
        m = G.Model(p, gpu); m.set_smoother(smoother)
        got = _stall(m, G, N, nl, over, m.set, m.get)
    m.close()
    assert got[0] == stats
    assert np.array_equal(got[1], psi)
    # the purpose of the case: nrelax climbed far (if the solver defaults move, find another stalling input)
    assert max(s[1] for s in stats) >= 50, stats


def test_schedule_refusals(gpu):
    """nrelax outside 2..100 (what mg_solve can produce) and modes without mode_pv_invert are refused, on one grid and on
    a group"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    kw = base_kw(64, 2)
    m = G.Model(G.make_params(**kw), gpu); m.set_smoother("rb")
    g = Group(G.make_params(**kw), 2, 1, 32, gpu, smoother="rb")
    for h, setf in ((m, m.set), (g, g.set_global)):
        setf(G.PSI, synth_psi(64, 2)); h.set_const()
        for bad, mode in (([1], -1), ([101], -1), ([4, 0], -1), ([], -1), ([4], 0), ([4], 2), ([4], -2)):
            with pytest.raises(G.MsqgError) as e:
                h.test_cycles(bad, mode)
            assert e.value.code == G.ERR_ARG
        assert h.test_cycles([2, 100]).shape == (2,)
    m.close(); g.close()
