"""Domain decomposition (reference -D_MPI=1 semantics) on ONE GPU with the local exchange back-end:
all tiles in one process, halo exchange by device copies.  Checked bit for bit against the oracle's
emulation of the MPI block decomposition (orc_set_decomp)."""
import numpy as np
import pytest

from common import base_kw, synth_psi

pytestmark = pytest.mark.gpu


def _pair(N, nl, px, py, agg_n, gpu):
    from oracle import oracle as O
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    kw = base_kw(N, nl)
    mo = O.Model(O.make_params(**kw))
    mo.L.orc_set_decomp(mo.h, px, py, agg_n)
    g = Group(G.make_params(**kw), px, py, agg_n, gpu)
    psi = synth_psi(N, nl)
    mo.set(O.PSI, psi)
    g.set_global(G.PSI, psi)
    mo.set_const(); g.set_const()
    return mo, g, psi


@pytest.mark.parametrize("N,nl,px,py,agg_n", [(128, 2, 2, 1, 32), (128, 3, 2, 2, 32), (256, 2, 4, 2, 64), (128, 4, 1, 2, 64)])
def test_decomposed_invertq_and_steps(gpu, N, nl, px, py, agg_n):
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, g, psi = _pair(N, nl, px, py, agg_n, gpu)
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); g.set_global(G.PSI, z)
    mo.invertq(); g.invertq()
    so, sg = mo.mgstats(), g.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI))
    for _ in range(3):
        assert g.step() == mo.step()
    assert g.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q))
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI))
    assert g.exchanges > 0


def test_decomposition_differs_from_serial_only_at_solver_tolerance(gpu):
    """block Gauss-Seidel is a different iterate from the serial sweep (poisson_layer.h:55-65) but the
    same solution to the solver tolerance"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N, nl = 128, 2
    kw = base_kw(N, nl)
    psi = synth_psi(N, nl)
    s = G.Model(G.make_params(**kw), gpu); s.set(G.PSI, psi); s.set_const()
    g = Group(G.make_params(**kw), 2, 2, 32, gpu); g.set_global(G.PSI, psi); g.set_const()
    for _ in range(2):
        s.step(); g.step()
    a, b = s.get(G.PSI), g.get_global(G.PSI)
    assert not np.array_equal(a, b)
    assert np.abs(a - b).max() < 1e-3 * np.abs(a).max()


@pytest.mark.parametrize("N,nl,px,py,agg_n,p2p", [(128, 2, 2, 1, 64, 1), (128, 3, 2, 2, 64, 1), (256, 2, 4, 2, 128, 1), (256, 4, 1, 2, 64, 1),
                                                   (512, 4, 4, 2, 256, 1), (256, 3, 2, 2, 64, 0), (256, 2, 4, 2, 128, 0),
                                                   # 2 and 1 fused sweeps per tile pass (nl 5-8, 9-12), both transports
                                                   (256, 7, 2, 2, 64, 1), (256, 12, 2, 1, 64, 1), (256, 9, 1, 2, 64, 0)])
def test_red_black_group_equals_single_gpu_and_oracle(gpu, N, nl, px, py, agg_n, p2p, monkeypatch):
    """Throughput mode on tiles: a red-black half-sweep does not depend on the decomposition, so the group (deep halos,
    one exchange per level, replicated coarse levels) must give the bits of the undecomposed solve and of the oracle
    running the same ordering -- including cold-start solves whose nrelax adapts upwards (several relax passes)."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    monkeypatch.setenv("MSQG_P2P", str(p2p))   # halo transport: stores into the neighbours' receive areas / staged copies
    kw = base_kw(N, nl)
    psi = synth_psi(N, nl)
    mo = O.Model(O.make_params(**kw)); mo.set_smoother("rb")
    s = G.Model(G.make_params(**kw), gpu); s.set_smoother("rb")
    g = Group(G.make_params(**kw), px, py, agg_n, gpu, smoother="rb")
    assert g.transport == ("peer-memory" if p2p else "nccl")
    mo.set(O.PSI, psi); s.set(G.PSI, psi); g.set_global(G.PSI, psi)
    mo.set_const(); s.set_const(); g.set_const()
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); s.set(G.PSI, z); g.set_global(G.PSI, z)
    mo.invertq(); s.invertq(); g.invertq()
    so, ss, sg = mo.mgstats(), s.mgstats(), g.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa) == (ss.i, ss.nrelax, ss.resb, ss.resa)
    assert np.array_equal(g.get_global(G.PSI), s.get(G.PSI))
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI))
    for _ in range(3):
        dt = g.step()
        assert dt == s.step() == mo.step()
    assert g.total_cycles == s.total_cycles == mo.L.orc_total_cycles(mo.h)
    for f, fo in ((G.Q, O.Q), (G.PSI, O.PSI)):
        assert np.array_equal(g.get_global(f), s.get(f))
        assert np.array_equal(g.get_global(f), mo.get(fo))
    assert g.exchanges > 0


def test_nccl_backend_two_gpus(gpu):
    """the NCCL back-end (one tile per process) under torchrun on 2 GPUs, both smoothers, bit-exact against the oracle;
    skipped on a single-GPU box"""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for sm in ("rb", "lex", "rbper"):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(root, "scripts", "dist_check.py"), sm],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "DIST_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
