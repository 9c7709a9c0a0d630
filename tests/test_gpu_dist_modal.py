"""The vertical-mode inversion (mode_pv_invert = 1) on red-black tiles.

Every mode is a scalar Helmholtz solve through the same deep-halo cycle as the layer-coupled problem, so the group must
give the bits of the single-GPU modal solve and of the oracle with the red-black ordering: psi, q, dt, the statistics of
every mode and the cycle counts, whatever the tiles, the halo transport, the relax kernel or graph replay."""
import os
import subprocess
import sys

import numpy as np
import pytest

from common import base_kw, synth_psi

pytestmark = pytest.mark.gpu


def _need_lapack():
    from oracle import oracle as O
    if O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")


CASES = [
    # N, nl, px, py, agg_n, p2p, environment, parameters, amplitude of psi
    (128, 2, 2, 1, 64, 1, {}, {}, 1.),
    (128, 3, 1, 2, 64, 0, {}, {}, 1.),
    (128, 4, 2, 2, 64, 1, {}, {}, 1.),
    (256, 3, 4, 2, 128, 1, {}, {}, 1.),
    (256, 2, 4, 2, 128, 0, {}, {}, 1.),
    (128, 10, 2, 2, 64, 1, {}, {}, 1.),                                # projections at NL = 10
    (128, 10, 2, 1, 64, 0, {}, {}, 1.),
    (128, 3, 2, 2, 64, 1, {"MSQG_RB_TILE": "0"}, {}, 1.),              # the streaming NL = 1 pass with a deep halo
    (128, 4, 1, 2, 64, 0, {"MSQG_RB_TILE": "0"}, {}, 1.),
    (128, 3, 2, 2, 64, 1, {"MSQG_GRAPH": "0"}, {}, 1.),                # eager launches
    (128, 3, 2, 1, 64, 0, {}, dict(Re=300., Eks=0.001), 1.),           # laplacian viscosity and surface Ekman friction
    # a residual at the round-off floor of a huge q: modes 0 and 1 stagnate for 100 cycles and nrelax climbs to about
    # 90, so every distributed level runs its sweeps in many exchange chunks of at most 7
    (128, 3, 2, 2, 64, 1, {}, {}, 1e13),
    (128, 3, 2, 1, 64, 0, {"MSQG_RB_TILE": "0"}, {}, 1e13),
]


@pytest.mark.parametrize("N,nl,px,py,agg_n,p2p,env,over,amp", CASES)
def test_modal_group_equals_single_gpu_and_oracle(gpu, N, nl, px, py, agg_n, p2p, env, over, amp, monkeypatch):
    from oracle import oracle as O
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    _need_lapack()
    monkeypatch.setenv("MSQG_P2P", str(p2p))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    kw = base_kw(N, nl, mode_pv_invert=1, **over)
    psi = amp * synth_psi(N, nl)
    mo = O.Model(O.make_params(**kw)); mo.set_smoother("rb")
    s = G.Model(G.make_params(**kw), gpu); s.set_smoother("rb")
    g = Group(G.make_params(**kw), px, py, agg_n, gpu, smoother="rb")
    assert g.transport == ("peer-memory" if p2p else "nccl")
    mo.set(O.PSI, psi); s.set(G.PSI, psi); g.set_global(G.PSI, psi)
    mo.set_const(); s.set_const(); g.set_const()
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q))

    def stats(m):
        return [(x.i, x.nrelax, x.resb, x.resa) for x in (m.mgstats(k) for k in range(nl))]

    # cold start: psi = 0 and the modal unknowns as allocated (0), nrelax adapts upwards
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); s.set(G.PSI, z); g.set_global(G.PSI, z)
    mo.invertq(); s.invertq(); g.invertq()
    cold = stats(g)
    assert cold == stats(s) == stats(mo)
    assert tuple(getattr(g.mgstats(), f) for f in ("i", "nrelax", "resb", "resa")) == cold[-1]
    assert np.array_equal(g.get_global(G.PSI), s.get(G.PSI))
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI))
    nrelax = {x[1] for x in cold}
    for _ in range(4 if amp == 1. else 2):
        dt = g.step()
        assert dt == s.step() == mo.step()
        nrelax |= {x[1] for x in stats(g)}
        assert stats(g) == stats(s) == stats(mo)
    assert g.total_cycles == s.total_cycles == mo.L.orc_total_cycles(mo.h)
    for f, fo in ((G.Q, O.Q), (G.PSI, O.PSI)):
        assert np.array_equal(g.get_global(f), s.get(f))
        assert np.array_equal(g.get_global(f), mo.get(fo))
    assert g.exchanges > 0
    print("modal %d^2 x %d on %dx%d (%s): nrelax reached %s, cycles %d, exchanges %d"
          % (N, nl, px, py, g.transport, sorted(nrelax), g.total_cycles, g.exchanges))
    g.close(); s.close()


def test_modal_group_refusals(gpu):
    """what the modal group does not build is refused with MSQG_ERR_ARG"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N, nl = 128, 3
    kw = base_kw(N, nl, mode_pv_invert=1)
    with pytest.raises(G.MsqgError, match="red-black") as e:
        Group(G.make_params(**kw), 2, 1, 64, gpu, smoother="lex")
    assert e.value.code == G.ERR_ARG
    with pytest.raises(G.MsqgError, match="varRo") as e:
        Group(G.make_params(**base_kw(N, nl, mode_pv_invert=1, varRo=1)), 2, 1, 64, gpu, smoother="rb")
    assert e.value.code == G.ERR_ARG
    with pytest.raises(G.MsqgError, match="stochastic") as e:
        Group(G.make_params(**base_kw(N, nl, stochastic=1, tr_stoch=10., amp_stoch=1.)), 2, 1, 64, gpu, smoother="rb")
    assert e.value.code == G.ERR_ARG


@pytest.mark.parametrize("px,py,split", [(2, 1, "x"), (2, 2, "y")])
def test_modal_group_refuses_fr_that_differs_between_tiles(gpu, px, py, split):
    """an Fr field constant on every tile but not across tiles gives every tile uniform modes of its own: refused"""
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    _need_lapack()
    N, nl = 128, 3
    kw = base_kw(N, nl, mode_pv_invert=1)
    fr = np.zeros((nl, N, N))
    for l in range(nl - 1):
        fr[l] = kw["Fr"][l]
    g = Group(G.make_params(**kw), px, py, 64, gpu, smoother="rb")
    g.set_global(G.PSI, synth_psi(N, nl))
    g.set_global(G.FR, fr)
    g.set_const()   # the same Fr everywhere, given as a field: accepted
    if split == "x":
        fr[1, :, N // 2:] *= 1.5
    else:
        fr[0, N // 2:, :] = np.nextafter(fr[0, N // 2:, :], 1.)   # one ulp is enough
    g.set_global(G.FR, fr)
    with pytest.raises(G.MsqgError, match="Fr of interface %d differs" % (1 if split == "x" else 0)) as e:
        g.set_const()
    assert e.value.code == G.ERR_ARG
    g.close()


def test_modal_nccl_backend_two_gpus(gpu):
    """the NCCL back-end (one tile per process) of the modal group under torchrun, bit-exact against the oracle;
    skipped on a single-GPU box"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _need_lapack()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29534", os.path.join(root, "scripts", "dist_check.py"), "rbmodal"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DIST_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
