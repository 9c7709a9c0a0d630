"""Doubly periodic boundaries, sbc = -1 (msqg/qg.h:80, :842-846: periodic(right); periodic(top), bc_type = -2).

On the GPU the periodic domain runs on the tile machinery of the multi-GPU path: every side of every tile is an internal
side whose halo comes from the tile across the seam -- the tile itself for px = 1 or py = 1 -- and the levels below
the tiles (up to 32^2 for nl <= 9, up to 16^2 for nl >= 10) are swept by the single-CTA coarse kernel with wrap-around
neighbours.  Red-black ordering only (a half-sweep does not
depend on where the seam is).  Bit-exact against the oracle, whose boundary() copies the opposite side into the ghost
ring on every level ([BASILISK] periodic box boundaries)."""
import numpy as np
import pytest

from common import base_kw, periodic_psi

pytestmark = pytest.mark.gpu


def _diff(a, b):
    d = np.abs(a - b)
    return "max |difference| %.3e at %d of %d cells" % (d.max(), int((d > 0).sum()), d.size)


@pytest.mark.parametrize("N,nl,px,py,over", [(64, 2, 1, 1, {}), (128, 3, 1, 1, dict(Re=200.)), (128, 4, 2, 1, {}), (128, 3, 2, 2, {}),
                                              (256, 2, 4, 2, dict(Eks=0.001)), (32, 3, 1, 1, {}), (64, 5, 1, 2, {}),
                                              # layer counts whose coarse kernel holds fewer levels (nl >= 10), and 2 or 1
                                              # fused sweeps per pass of the tile relaxation (nl 5-8, 9-12)
                                              (64, 10, 1, 1, {}), (128, 12, 2, 1, {}), (64, 11, 2, 2, {}), (128, 6, 1, 1, {}),
                                              (128, 7, 2, 2, {}), (64, 8, 1, 2, {}), (128, 9, 2, 1, {})])
def test_periodic_domain_matches_oracle(gpu, N, nl, px, py, over):
    from oracle import oracle as O
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    kw = base_kw(N, nl, sbc=-1., **over)
    psi = periodic_psi(N, nl)
    mo = O.Model(O.make_params(**kw)); mo.set_smoother("rb")
    g = Group(G.make_params(**kw), px, py, 0, gpu, smoother="rb")
    mo.set(O.PSI, psi); g.set_global(G.PSI, psi)
    mo.set_const(); g.set_const()
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q)), "q: " + _diff(g.get_global(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); g.set_global(G.PSI, z)
    mo.invertq(); g.invertq()
    so, sg = mo.mgstats(), g.mgstats()
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI)), "psi after invertq: " + _diff(g.get_global(G.PSI), mo.get(O.PSI))
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
    mo.set(O.PSI, psi); g.set_global(G.PSI, psi)
    for _ in range(4):
        assert g.step() == mo.step()
    assert g.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(g.get_global(G.Q), mo.get(O.Q)), "q: " + _diff(g.get_global(G.Q), mo.get(O.Q))
    assert np.array_equal(g.get_global(G.PSI), mo.get(O.PSI)), "psi: " + _diff(g.get_global(G.PSI), mo.get(O.PSI))
    # periodic and closed-basin runs of the same initial state differ from the first step on
    kw2 = base_kw(N, nl, **over)
    mc = O.Model(O.make_params(**kw2)); mc.set_smoother("rb")
    mc.set(O.PSI, psi); mc.set_const()
    assert not np.array_equal(mc.get(O.Q), mo.get(O.Q))


def test_periodic_through_the_single_model_entry_points(gpu):
    """msqg_create with sbc = -1 hands out the tile of a 1 x 1 periodic group: set_const / invertq / update / advance /
    step of the plain C ABI (and with it qg.e and the python module) work unchanged; the plugin sequence
    update -> advance equals the fused step, as on a closed basin."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    N, nl = 64, 3
    kw = base_kw(N, nl, sbc=-1.)
    psi = periodic_psi(N, nl)
    mo = O.Model(O.make_params(**kw)); mo.set_smoother("rb")
    import torch
    mg = G.Model(G.make_params(**kw), gpu)
    assert mg.L.msqg_get_smoother(mg.h) == 1
    st = torch.cuda.Stream(device=gpu)   # a caller's stream (bench.py does this): the group behind the handle follows
    mg.set_stream(st.cuda_stream)
    with pytest.raises(G.MsqgError):
        mg.set_smoother("lex")
    mo.set(O.PSI, psi); mg.set(G.PSI, psi)
    mo.set_const(); mg.set_const()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))
    assert mg.update(1e10) == mo.update(1e10)
    assert np.array_equal(mg.get(G.DQ), mo.get(O.DQ))
    for _ in range(3):
        assert mg.step() == mo.step()
    so, sg = mo.mgstats(), mg.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    # q -> psi -> q round trip through the entry points the python module uses (pyq2p / pyp2q)
    mg.invertq(); mg.comp_q(); mo.invertq(); mo.comp_q()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))


def test_periodic_rejects_what_is_not_built(gpu):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    with pytest.raises(G.MsqgError):
        Group(G.make_params(**base_kw(64, 2, sbc=-1.)), 1, 1, 0, gpu, smoother="lex")
    with pytest.raises(G.MsqgError):
        G.Model(G.make_params(**base_kw(64, 2, sbc=-1., upg=[0.1, 0.], vpg=[0., 0.])), gpu)
    with pytest.raises(G.MsqgError):
        G.Model(G.make_params(**base_kw(64, 2, sbc=-1., mode_pv_invert=1)), gpu)
    # the wrap-around coarse kernel holds levels up to 32^2 for nl <= 9 but only up to 16^2 for nl >= 10: from nl = 10 on
    # the tiles start at the 32^2 level, which 4 tiles across cannot split into the 16 cells a red-black tile needs
    Group(G.make_params(**base_kw(128, 9, sbc=-1.)), 4, 2, 0, gpu, smoother="rb").close()
    with pytest.raises(G.MsqgError, match="periodic"):
        Group(G.make_params(**base_kw(128, 10, sbc=-1.)), 4, 2, 0, gpu, smoother="rb")
    with pytest.raises(G.MsqgError, match="periodic"):
        Group(G.make_params(**base_kw(128, 12, sbc=-1.)), 2, 4, 0, gpu, smoother="rb")


def test_periodic_full_size_translation_equivariance(gpu):
    """2048^2 x 4, where the oracle is too slow: the periodic step commutes BIT FOR BIT with a diagonal shift by N/2 cells
    (constant coefficients once the wind is off; the hierarchy down to 2 x 2 cells maps onto itself; red-black
    half-sweeps do not depend on traversal order) -- the property tests/test_oracle_rb.py pins on the oracle, here across
    hundreds of CTAs, the wrap-around halos of every level and the recorded cycle graphs."""
    from msom_b200 import capi as G
    N, nl = 2048, 4
    psi = periodic_psi(N, nl)
    sh = lambda a: np.roll(a, (N // 2, N // 2), axis=(1, 2))

    def run(p0, nsteps=3):
        m = G.Model(G.make_params(**base_kw(N, nl, sbc=-1., tau0=0.)), gpu)
        m.set(G.PSI, p0); m.set_const()
        q0 = m.get(G.Q)
        dts = [m.step() for _ in range(nsteps)]
        out = (q0, m.get(G.Q), m.get(G.PSI), dts, m.total_cycles)
        m.close()
        return out

    q0, q1, p1, dts, cyc = run(psi)
    r0, r1, rp, rdts, rcyc = run(sh(psi))
    assert rdts == dts and rcyc == cyc and cyc >= 6
    assert np.array_equal(r0, sh(q0)) and np.array_equal(r1, sh(q1)) and np.array_equal(rp, sh(p1))
    assert np.isfinite(q1).all() and not np.array_equal(q1, q0)
