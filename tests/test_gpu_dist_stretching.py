"""Horizontally varying stretching (varRo > 0: Ro(y), msqg/qg.h:1032-1037; a Fr(x, y) field: qg.h:957-962) on red-black
tile groups and on the doubly periodic domain.

The group decides constants / per-row tables / per-cell tables once for all tiles (msqg_group_set_const), builds the
tables of every tile over its own cells plus the halo its sweeps reach, and gathers the stretching onto the solver tile
for the coarse levels.  So the group must give the bits of the undecomposed red-black model and of the oracle's
red-black ordering: q, psi, dt, the solver statistics and the cycle counts, whatever the tiles, the halo transport, the
relax kernel or graph replay."""
import os
import subprocess
import sys

import numpy as np
import pytest

from common import base_kw, periodic_psi, synth_psi

pytestmark = pytest.mark.gpu


def _fr_field(N, nl):
    """the Fr(x, y) field of test_gpu_variants.test_stretching_varies_in_x_and_y"""
    rng = np.random.default_rng(77)
    y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
    fr = np.zeros((nl, N, N))
    for l in range(nl - 1):
        fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y) + 0.05 * rng.uniform(-1, 1, (N, N)))
    return fr


def _setup(stretch, N, nl, over):
    """parameters and Fr field of a stretching case: rows = varRo, cells = Fr(x, y), both = the two together"""
    kw = base_kw(N, nl, **over)
    if stretch in ("rows", "both"):
        kw["varRo"] = 1
    fr = _fr_field(N, nl) if stretch in ("cells", "both") else None
    return kw, fr, ("rows" if stretch == "rows" else "cells")


def _run_three(kw, fr, psi, make_group, gpu, nsteps=3):
    """oracle (rb), undecomposed model (rb) and the group from the same inputs; set_const, cold-start invertq, steps"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo = O.Model(O.make_params(**kw)); mo.set_smoother("rb")
    s = G.Model(G.make_params(**kw), gpu); s.set_smoother("rb")
    g = make_group()
    mo.set(O.PSI, psi); s.set(G.PSI, psi); g.set_global(G.PSI, psi)
    if fr is not None:
        mo.set(O.FR, fr); s.set(G.FR, fr); g.set_global(G.FR, fr)
    mo.set_const(); s.set_const(); g.set_const()
    assert np.array_equal(g.get_global(G.Q), s.get(G.Q))
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); s.set(G.PSI, z); g.set_global(G.PSI, z)
    mo.invertq(); s.invertq(); g.invertq()
    so, ss, sg = mo.mgstats(), s.mgstats(), g.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa) == (ss.i, ss.nrelax, ss.resb, ss.resa)
    assert np.array_equal(g.get_global(G.PSI), s.get(G.PSI))
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI))
    nrelax = {sg.nrelax}
    for _ in range(nsteps):
        dt = g.step()
        assert dt == s.step() == mo.step()
        so, ss, sg = mo.mgstats(), s.mgstats(), g.mgstats()
        assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa) == (ss.i, ss.nrelax, ss.resb, ss.resa)
        nrelax.add(sg.nrelax)
    assert g.total_cycles == s.total_cycles == mo.L.orc_total_cycles(mo.h)
    for f, fo in ((G.Q, O.Q), (G.PSI, O.PSI)):
        assert np.array_equal(g.get_global(f), s.get(f))
        assert np.array_equal(g.get_global(f), mo.get(fo))
    return mo, s, g, nrelax


CASES = [
    # N, nl, px, py, agg_n, p2p, stretching, environment, parameters
    (128, 2, 2, 1, 64, 1, "rows", {}, {}),
    (128, 3, 1, 2, 64, 0, "cells", {}, {}),
    (128, 4, 2, 2, 32, 1, "both", {}, {}),        # agg_n 32: every gathered level inside k_coarse_rb
    (256, 3, 4, 2, 128, 1, "cells", {}, {}),      # agg_n 128: level 64^2 on the solver tile outside k_coarse_rb
    (256, 2, 4, 2, 128, 0, "rows", {}, {}),
    (512, 3, 4, 2, 128, 1, "both", {}, {}),       # larger tiles on 4 x 2
    (256, 5, 2, 2, 64, 1, "rows", {}, {}),        # nl 5-6: the streaming kernel (2 fused sweeps per pass)
    (128, 6, 2, 1, 64, 0, "cells", {}, {}),
    (256, 6, 1, 2, 128, 1, "both", {}, {}),
    (128, 3, 2, 2, 64, 1, "cells", {"MSQG_RB_TILE": "0"}, {}),              # the streaming kernel at nl <= 4
    (128, 4, 1, 2, 64, 0, "both", {"MSQG_RB_COARSE_TABLES": "0"}, {}),     # tables through level-by-level launches
    (128, 2, 2, 2, 64, 1, "rows", {"MSQG_GRAPH": "0"}, {}),                # eager launches
    (128, 3, 2, 1, 64, 1, "both", {}, dict(Re=300.)),                      # laplacian viscosity
]


@pytest.mark.parametrize("N,nl,px,py,agg_n,p2p,stretch,env,over", CASES)
def test_group_varying_stretching_equals_single_gpu_and_oracle(gpu, N, nl, px, py, agg_n, p2p, stretch, env, over, monkeypatch):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    monkeypatch.setenv("MSQG_P2P", str(p2p))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    kw, fr, want = _setup(stretch, N, nl, over)
    make = lambda: Group(G.make_params(**kw), px, py, agg_n, gpu, smoother="rb")
    mo, s, g, nrelax = _run_three(kw, fr, synth_psi(N, nl), make, gpu)
    assert g.transport == ("peer-memory" if p2p else "nccl")
    assert g.stretching == s.stretching == want
    assert g.exchanges > 0
    g.close(); s.close()


@pytest.mark.parametrize("N,nl,px,py,p2p,stretch", [(128, 3, 2, 2, 1, "cells"),   # tile kernel
                                                     (128, 5, 2, 1, 0, "rows")])  # streaming kernel
def test_group_varying_stretching_stalled_solve(gpu, N, nl, px, py, p2p, stretch, monkeypatch):
    """a residual at the round-off floor of a huge q: nrelax climbs far above 7, so every distributed level runs its
    sweeps in several exchange chunks, each reading the tables deep into the halo"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    monkeypatch.setenv("MSQG_P2P", str(p2p))
    kw, fr, want = _setup(stretch, N, nl, {})
    make = lambda: Group(G.make_params(**kw), px, py, 64, gpu, smoother="rb")
    mo, s, g, nrelax = _run_three(kw, fr, 1e13 * synth_psi(N, nl), make, gpu, nsteps=2)
    assert max(nrelax) > 7
    assert g.stretching == want
    print("stalled %s %d^2 x %d on %dx%d: nrelax reached %s" % (stretch, N, nl, px, py, sorted(nrelax)))
    g.close(); s.close()


SCHED = [2, 3, 4, 5, 6, 7, 8, 9, 13, 16, 17, 100]


@pytest.mark.parametrize("stretch,nl,px,py", [("rows", 3, 2, 2), ("cells", 4, 2, 1), ("cells", 5, 1, 2)])
def test_group_fixed_schedules(gpu, stretch, nl, px, py):
    """msqg_group_test_cycles with every sweep count of a fixed schedule equals the undecomposed model's cycles"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N = 128
    kw, fr, want = _setup(stretch, N, nl, {})
    psi = synth_psi(N, nl)
    s = G.Model(G.make_params(**kw), gpu); s.set_smoother("rb")
    g = Group(G.make_params(**kw), px, py, 64, gpu, smoother="rb")
    for setf in (s.set, g.set_global):
        setf(G.PSI, psi)
        if fr is not None:
            setf(G.FR, fr)
    s.set_const(); g.set_const()
    z = np.zeros_like(psi)
    s.set(G.PSI, z); g.set_global(G.PSI, z)
    ra, rb = s.test_cycles(SCHED), g.test_cycles(SCHED)
    assert np.array_equal(rb, ra)
    assert np.array_equal(g.get_global(G.PSI), s.get(G.PSI))
    assert g.stretching == want
    g.close(); s.close()


@pytest.mark.parametrize("px,py,split", [(2, 1, "x"), (2, 2, "x"), (1, 2, "y"), (2, 2, "y")])
def test_fr_constant_per_tile_but_not_across_tiles(gpu, px, py, split):
    """Fr constant on every tile but different between tiles: each tile alone sees uniform stretching, the field is not.
    The group takes the path of the undecomposed model (tables) and gives its bits."""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N, nl = 128, 3
    kw = base_kw(N, nl)
    fr = np.zeros((nl, N, N))
    for l in range(nl - 1):
        fr[l] = kw["Fr"][l]
    if split == "x":   # left and right halves differ: every row holds two values
        fr[1, :, N // 2:] *= 1.5
    else:              # bottom and top halves differ: the field still only varies with y
        fr[0, N // 2:, :] *= 1.25

    make = lambda: Group(G.make_params(**kw), px, py, 64, gpu, smoother="rb")
    mo, s, g, _ = _run_three(kw, fr, synth_psi(N, nl), make, gpu)
    assert g.stretching == s.stretching == ("cells" if split == "x" else "rows")
    g.close(); s.close()


@pytest.mark.parametrize("nl,px,py,stretch", [(2, 1, 1, "cells"), (3, 1, 1, "rows"), (4, 2, 1, "both"), (3, 2, 2, "cells"),
                                              (5, 2, 2, "rows"), (6, 1, 1, "both"), (6, 2, 1, "cells"), (5, 1, 2, "both")])
def test_periodic_varying_stretching_matches_oracle(gpu, nl, px, py, stretch):
    """sbc = -1: the 1 x 1 periodic group behind a G.Model handle and periodic groups, against the oracle (which applies
    the periodic boundary to Frl / strl)"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N = 128
    kw, fr, want = _setup(stretch, N, nl, dict(sbc=-1.))
    psi = periodic_psi(N, nl)
    mo = O.Model(O.make_params(**kw)); mo.set_smoother("rb")
    g = G.Model(G.make_params(**kw), gpu) if px * py == 1 else Group(G.make_params(**kw), px, py, 0, gpu, smoother="rb")
    setg = g.set if px * py == 1 else g.set_global
    getg = g.get if px * py == 1 else g.get_global
    mo.set(O.PSI, psi); setg(G.PSI, psi)
    if fr is not None:
        mo.set(O.FR, fr); setg(G.FR, fr)
    mo.set_const(); g.set_const()
    assert g.stretching == want
    assert np.array_equal(getg(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); setg(G.PSI, z)
    mo.invertq(); g.invertq()
    so, sg = mo.mgstats(), g.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
    assert np.array_equal(getg(G.PSI), mo.get(O.PSI))
    mo.set(O.PSI, psi); setg(G.PSI, psi)
    for _ in range(3):
        assert g.step() == mo.step()
    assert g.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(getg(G.Q), mo.get(O.Q)) and np.array_equal(getg(G.PSI), mo.get(O.PSI))
    g.close()


def test_varying_stretching_refusals(gpu, monkeypatch):
    """what stays unbuilt is refused with MSQG_ERR_ARG at the first solve"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N = 128

    def refused(g, match):
        with pytest.raises(G.MsqgError, match=match) as e:
            g.invertq()
        assert e.value.code == G.ERR_ARG

    # the lexicographic (reference-order) group has no tiled sweep with coefficient tables
    g = Group(G.make_params(**base_kw(N, 3, varRo=1)), 2, 1, 64, gpu, smoother="lex")
    g.set_global(G.PSI, synth_psi(N, 3)); g.set_const()
    assert g.stretching == "rows"
    refused(g, "red-black")
    with pytest.raises(G.MsqgError, match="red-black"):
        g.test_cycles([4])
    g.close()
    # the layer-coupled tables are built for nl <= 6, as on one GPU
    g = Group(G.make_params(**base_kw(N, 7, varRo=1)), 2, 2, 64, gpu, smoother="rb")
    g.set_global(G.PSI, synth_psi(N, 7)); g.set_const()
    refused(g, "nl <= 6")
    g.close()
    # periodic: every replicated level must be swept by k_coarse_rb, which reads the tables only when allowed to
    monkeypatch.setenv("MSQG_RB_COARSE_TABLES", "0")
    m = G.Model(G.make_params(**base_kw(64, 3, sbc=-1., varRo=1)), gpu)
    m.set(G.PSI, periodic_psi(64, 3)); m.set_const()
    refused(m, "periodic")
    m.close()


def test_uniform_stretching_reports_uniform(gpu):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N, nl = 128, 3
    kw = base_kw(N, nl)
    m = G.Model(G.make_params(**kw), gpu)
    with pytest.raises(G.MsqgError):
        m.stretching   # decided by set_const
    m.set(G.PSI, synth_psi(N, nl)); m.set_const()
    assert m.stretching == "uniform"
    for sm in ("rb", "lex"):
        g = Group(G.make_params(**kw), 2, 2, 64, gpu, smoother=sm)
        fr = np.zeros((nl, N, N))
        for l in range(nl - 1):
            fr[l] = kw["Fr"][l]
        g.set_global(G.PSI, synth_psi(N, nl)); g.set_global(G.FR, fr); g.set_const()
        assert g.stretching == "uniform"
        g.close()
    m.close()


def test_varying_stretching_nccl_two_gpus(gpu):
    """the NCCL back-end (one tile per process) with varRo and a per-cell Fr field, bit-exact against the oracle on
    every rank; skipped on a single-GPU box"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29537", os.path.join(root, "scripts", "dist_check.py"), "rbvary"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DIST_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
