"""GPU parity of the whole path (set_const, invertq, update_qg, the RK2 step)
against the CPU oracle through the C ABI.  north_star tolerances: relative L2
of psi and q <= 1e-12 after one step, <= 1e-9 after 100 steps, equal multigrid
cycle counts; the implementation is in fact bit-identical."""
import numpy as np
import pytest

from common import make_pair, rel_l2

pytestmark = pytest.mark.gpu


NL_HIGH = range(5, 13)   # every layer count of the reference-order relax kernel above the common ones


@pytest.mark.parametrize("N,nl", [(64, 2), (256, 2), (128, 3), (128, 4), (64, 10)] + [(256, nl) for nl in NL_HIGH])
def test_set_const_and_invertq(gpu, N, nl):
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, psi = make_pair(N, nl)
    mo.set_const(); mg.set_const()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))          # comp_q
    assert np.array_equal(mg.get(G.STR)[: nl - 1], mo.get(O.STR)[: nl - 1])
    # cold start: psi = 0, several cycles with nrelax adaptation
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()
    so, sg = mo.mgstats(), mg.mgstats()
    assert (sg.i, sg.nrelax) == (so.i, so.nrelax)
    assert sg.resb == so.resb and sg.resa == so.resa
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))


@pytest.mark.parametrize("N,nl", [(256, 2), (128, 3), (128, 4)])
def test_update_qg(gpu, N, nl):
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(N, nl)
    mo.set_const(); mg.set_const()
    dto = mo.update(mo.p.DT)
    dtg = mg.update(mg.p.DT)
    assert dtg == dto
    assert np.array_equal(mg.get(G.ZETA), mo.get(O.ZETA))
    assert np.array_equal(mg.get(G.DQ), mo.get(O.DQ))


@pytest.mark.parametrize("N,nl,nsteps", [(256, 2, 1), (256, 2, 100), (128, 3, 20), (128, 4, 20)] + [(256, nl, 3) for nl in NL_HIGH])
def test_steps(gpu, N, nl, nsteps):
    """BASELINE config 1 (256^2 x 2): 1 and 100 steps."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(N, nl)
    mo.set_const(); mg.set_const()
    for _ in range(nsteps):
        dto = mo.step()
        dtg = mg.step()
        assert dtg == dto
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)     # equal multigrid iteration counts
    tol = 1e-12 if nsteps == 1 else 1e-9
    for fg, fo in ((G.PSI, O.PSI), (G.Q, O.Q)):
        a, b = mg.get(fg), mo.get(fo)
        assert rel_l2(a, b) <= tol
        assert np.array_equal(a, b)                           # in fact bit-identical


def test_viscous_and_pg_terms(gpu):
    """Re, Re4, Eks, background flow (upg/vpg), flsrv, q_forc, topography all on."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    N, nl = 64, 3
    over = dict(Re=500., Eks=0.001, flsrv=1, upg=[0.1, 0.05, 0.0], vpg=[0.02, 0.0, -0.01])
    mo, mg, psi = make_pair(N, nl, **over)
    rng = np.random.default_rng(2)
    qf = 1e-3 * rng.standard_normal((nl, N, N))
    topo = 0.1 * rng.standard_normal((1, N, N))
    mo.set(O.QFORC, qf); mg.set(G.QFORC, qf)
    mo.set(O.TOPO, topo); mg.set(G.TOPO, topo)
    mo.L.orc_set_flag_topo(mo.h, 1); G.check(mg.L.msqg_set_flag_topo(mg.h, 1))
    mo.set_const(); mg.set_const()
    assert mg.update(mg.p.DT) == mo.update(mo.p.DT)
    assert np.array_equal(mg.get(G.DQ), mo.get(O.DQ))
    for _ in range(3):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))


@pytest.mark.parametrize("N,nl", [(8, 2), (16, 3), (32, 4), (64, 5), (64, 7), (32, 12), (16, 12)])
def test_edge_shapes(gpu, N, nl):
    """Smallest grids (one partial tile in every tiled kernel, a handful of strips in the relax wavefront) and layer
    counts up to the maximum the kernels are instantiated for (nl = 12): three steps bit-identical to the oracle,
    equal dt and equal multigrid cycle counts."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    over = {}
    if nl not in (2, 3, 4, 10):
        over = dict(dh=[1.0 / nl] * nl, Fr=list(np.linspace(0.002, 0.008, nl - 1)))
    mo, mg, _ = make_pair(N, nl, **over)
    mo.set_const(); mg.set_const()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))
    for _ in range(3):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)


def test_pipelined_field_io_equals_set_step_get(gpu):
    """msqg_set_field_async / _commit / msqg_get_field_async (include/msqg.h): a stream of independent states stepped with
    the uploads and downloads on their own streams gives the bits of msqg_set_field; step; msqg_get_field for every state,
    whatever the overlap; a third upload without a commit is refused."""
    import torch
    from common import base_kw, synth_psi
    from msom_b200 import capi as G
    N, nl, nstates = 128, 3, 5

    def model():
        mm = G.Model(G.make_params(**base_kw(N, nl)), gpu)
        mm.set_smoother("rb")
        mm.set(G.PSI, synth_psi(N, nl)); mm.set_const()
        return mm

    ms, m = model(), model()               # two identical models: warm starts and the dt chain evolve alike
    rng = np.random.default_rng(3)
    q0 = m.get(G.Q)
    states = [q0 * (1 + 0.05 * k) + 1e-3 * rng.standard_normal(q0.shape) for k in range(nstates)]
    ref = []
    for s in states:                       # serial: msqg_set_field; step; msqg_get_field
        ms.set(G.Q, s); ms.step(); ref.append(ms.get(G.Q))
    hin = [torch.empty(q0.shape, dtype=torch.float64).pin_memory() for _ in range(2)]
    hout = [torch.empty(q0.shape, dtype=torch.float64).pin_memory() for _ in range(nstates)]
    hin[0].copy_(torch.from_numpy(states[0]))
    m.set_async(G.Q, hin[0].numpy())
    for k in range(nstates):
        m.commit()
        if k + 1 < nstates:
            m.io_wait() if k >= 1 else None          # the other input buffer is about to be rewritten on the host
            hin[(k + 1) & 1].copy_(torch.from_numpy(states[k + 1]))
            m.set_async(G.Q, hin[(k + 1) & 1].numpy())
        m.step()
        m.get_async(G.Q, hout[k].numpy())
    m.io_wait()
    for k in range(nstates):
        assert np.array_equal(hout[k].numpy(), ref[k]), k
    m.set_async(G.Q, hin[0].numpy()); m.set_async(G.Q, hin[1].numpy())
    with pytest.raises(G.MsqgError):
        m.set_async(G.Q, hin[0].numpy())
    m.commit(); m.commit(); m.io_wait()
    with pytest.raises(G.MsqgError):
        m.set_async(G.FR, hin[0].numpy())
