"""GPU parity of the compile-time variants of the reference, exposed as runtime knobs:
MODE_PV_INVERT 1 (modal inversion through eigmode.h, BASELINE config 3) and
-D_STOCHASTIC=1 (qg_stochastic.h, BASELINE config 5); plus size-independent
properties at the full BASELINE shapes where the CPU oracle is too slow."""
import ctypes as C
import os

import numpy as np
import pytest

from common import base_kw, make_pair, rel_l2, synth_psi

pytestmark = pytest.mark.gpu
libc = C.CDLL(None)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("N,nl,nsteps", [(64, 2, 3), (128, 3, 5), (64, 10, 3)])
def test_modal_inversion(gpu, N, nl, nsteps):
    from oracle import oracle as O
    from msom_b200 import capi as G
    if O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")
    mo, mg, psi = make_pair(N, nl, mode_pv_invert=1)
    mo.set_const(); mg.set_const()
    for fid_g, fid_o in ((G.IBU, O.IBU), (G.CL2M, O.CL2M), (G.CM2L, O.CM2L), (G.Q, O.Q)):
        assert np.array_equal(mg.get(fid_g), mo.get(fid_o))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()
    for mode in range(nl):
        so, sg = mo.mgstats(mode), mg.mgstats(mode)
        assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa), mode
    assert np.array_equal(mg.get(G.PM), mo.get(O.PM))
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    for _ in range(nsteps):
        assert mg.step() == mo.step()
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI)) and np.array_equal(mg.get(G.Q), mo.get(O.Q))


@pytest.mark.parametrize("smoother", ["lex", "rb"])
@pytest.mark.parametrize("N,nl,varRo,frfield,nsteps", [(64, 2, 1, 0, 3), (64, 3, 0, 1, 3), (128, 3, 1, 1, 2), (32, 5, 1, 1, 2)])
def test_modal_inversion_varying_modes(gpu, N, nl, varRo, frfield, nsteps, smoother):
    """MODE_PV_INVERT 1 with horizontally varying Fr / Ro: the reference runs dgeev in every column (eigmode.h:74-299),
    so the projection matrices cl2m / cm2l and lambda = iBu are FIELDS; poisson() restricts lambda to every level
    ([BASILISK] restriction({alpha, lambda})) and relax() divides by -lambda[]*sq(Delta) + 4 cell by cell.  Bit-exact
    against the oracle in both sweep orders, equal cycle counts in every mode."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    if O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")
    mo, mg, psi = make_pair(N, nl, smoother=smoother, mode_pv_invert=1, varRo=varRo)
    if frfield:
        rng = np.random.default_rng(78)
        y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
        fr = np.zeros_like(psi)
        for l in range(nl - 1):
            fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y) + 0.05 * rng.uniform(-1, 1, (N, N)))
        mo.set(O.FR, fr); mg.set(G.FR, fr)
    mo.set_const(); mg.set_const()
    ibu = mo.get(O.IBU)
    assert np.ptp(ibu[1]) > 0                                   # the modes do vary
    for fid_g, fid_o in ((G.IBU, O.IBU), (G.CL2M, O.CL2M), (G.CM2L, O.CM2L), (G.Q, O.Q)):
        assert np.array_equal(mg.get(fid_g), mo.get(fid_o))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()
    for mode in range(nl):
        so, sg = mo.mgstats(mode), mg.mgstats(mode)
        assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa), mode
    assert np.array_equal(mg.get(G.PM), mo.get(O.PM))
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    for _ in range(nsteps):
        assert mg.step() == mo.step()
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI)) and np.array_equal(mg.get(G.Q), mo.get(O.Q))


@pytest.mark.parametrize("N,nl,nsteps", [(64, 3, 4), (32, 2, 6)])
def test_stochastic_forcing(gpu, N, nl, nsteps):
    """qg_stochastic.h: noise on libc rand() in the reference traversal order, float dts, relaxation term,
    no J(psi,zeta) in the top layer.  Both sides replay the same rand() stream (same seed, run in turn)."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    over = dict(stochastic=1, tr_stoch=10., amp_stoch=1.)
    mo, mg, _ = make_pair(N, nl, **over)
    sig = np.full((nl, N, N), 1e-3)
    mo.set(O.SSTOCH, sig); mg.set(G.SSTOCH, sig)
    mo.set_const(); mg.set_const()
    libc.srand(1000)                      # the oracle draws from the process-wide rand() like the reference
    dto = [mo.step() for _ in range(nsteps)]
    mg.L.msqg_seed_noise(mg.h, 1000)      # the GPU model owns a random_r state seeded like srand(1000)
    dtg = [mg.step() for _ in range(nsteps)]
    assert dtg == dto
    assert np.array_equal(mg.get(G.NSTOCH), mo.get(O.NSTOCH))
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    # the noise really entered q
    mo2, _, _ = make_pair(N, nl)
    mo2.set_const()
    for _ in range(nsteps):
        mo2.step()
    assert rel_l2(mo.get(O.Q), mo2.get(O.Q)) > 1e-8


@pytest.mark.parametrize("smoother", ["lex", "rb"])
def test_stochastic_forcing_philox(gpu, smoother):
    """production noise mode: Philox4x32-10 + Box-Muller on the device against the oracle's restatement of the same
    generator.  The integer stream is identical; log/cos of the CUDA math library and glibc may differ in the last
    place, so the noise field is compared to 1e-13 relative and the state after 4 steps to 1e-10."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    N, nl, nsteps = 64, 3, 4
    over = dict(stochastic=1, tr_stoch=10., amp_stoch=1.)
    mo, mg, _ = make_pair(N, nl, smoother=smoother, **over)
    sig = np.full((nl, N, N), 1e-3) * (1 + np.arange(nl)[:, None, None])
    mo.set(O.SSTOCH, sig); mg.set(G.SSTOCH, sig)
    mo.set_const(); mg.set_const()
    mo.L.orc_set_noise_mode(mo.h, 1, 4242)
    mg.L.msqg_seed_noise(mg.h, 4242); G.check(mg.L.msqg_set_noise_mode(mg.h, 1))
    for _ in range(nsteps):
        assert abs(mg.step() - mo.step()) <= 1e-15
    a, b = mg.get(G.NSTOCH), mo.get(O.NSTOCH)
    assert np.abs(a - b).max() <= 1e-13 * np.abs(b).max() and np.abs(b).max() > 0
    assert abs(b.mean()) < 5 * b.std() / np.sqrt(b.size)      # N(0, sigma): mean compatible with 0
    assert abs((b[0] / sig[0]).std() - 1) < 0.05               # unit variance before scaling
    for fg, fo in ((G.Q, O.Q), (G.PSI, O.PSI)):
        assert rel_l2(mg.get(fg), mo.get(fo)) <= 1e-10


def test_plugin_sequence_equals_fused_step(gpu):
    """update_qg / advance_qg called as the predictor-corrector does (msqg/qg.h:922-923 plugin surface)
    give the same bits as the fused msqg_step."""
    from msom_b200 import capi as G
    N, nl = 128, 3
    kw = base_kw(N, nl)
    a, b = G.Model(G.make_params(**kw), gpu), G.Model(G.make_params(**kw), gpu)
    psi = synth_psi(N, nl)
    for m in (a, b):
        m.set(G.PSI, psi); m.set_const()
    for _ in range(3):
        dt = a.update(a.p.DT, G.Q)               # dt = update(evolving, updates, DT)
        a.advance(G.QPRED, G.Q, dt / 2.)         # advance(predictor, evolving, updates, dt/2)
        a.update(dt, G.QPRED)                    # update(predictor, updates, dt)
        a.advance(G.Q, G.Q, dt)                  # advance(evolving, evolving, updates, dt)
        assert b.step() == dt
    assert np.array_equal(a.get(G.Q), b.get(G.Q)) and np.array_equal(a.get(G.PSI), b.get(G.PSI))


@pytest.mark.parametrize("N,nl,modal", [(1024, 3, 0), (2048, 10, 1), (4096, 4, 0)])
def test_full_size_properties(gpu, N, nl, modal):
    """BASELINE configs 2, 3 and the metric shape: q -> psi -> q round trip within the solver tolerance,
    residual statistic consistent, dt ramp of timestep() (DT/11 first), finite fields after a step."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    if modal and O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev")
    m = G.Model(G.make_params(**base_kw(N, nl, mode_pv_invert=modal)), gpu)
    rng = np.random.default_rng(5)
    psi = synth_psi(N, nl)
    m.set(G.PSI, psi); m.set_const()
    q0 = m.get(G.Q)
    G.check(m.L.msqg_reset_field(m.h, G.PSI))
    m.invertq()
    s = m.mgstats(nl - 1 if modal else -1)
    assert s.resa <= 1e-3 and 1 <= s.i < 100
    m.comp_q()
    err = np.abs(m.get(G.Q) - q0).max()
    if not modal:
        assert err == pytest.approx(s.resa, rel=1e-6)     # max|q - L(psi)| is exactly the reported residual
    assert err <= 1e-3 * nl * 4                            # modal: sum over modes of per-mode residuals
    m.set(G.Q, q0)
    dt = m.step()
    assert dt == pytest.approx(m.p.DT / 11, rel=1e-12)
    assert np.isfinite(m.get(G.Q)).all() and np.isfinite(m.get(G.PSI)).all()
    del rng


def test_ensemble_members_concurrent(gpu):
    """BASELINE config 5 in miniature: stochastic members batched on one GPU (own streams, own rand() replay)
    give, member by member, the bits of the same member run alone and of the oracle."""
    import time
    from oracle import oracle as O
    from msom_b200 import capi as G
    from msom_b200.ensemble import Ensemble
    N, nl, nmem, nsteps = 64, 3, 4, 3
    kw = base_kw(N, nl, stochastic=1, tr_stoch=10., amp_stoch=1.)
    sig = np.full((nl, N, N), 1e-3)
    psi = synth_psi(N, nl)
    ens = Ensemble(G.make_params(**kw), nmem, gpu)
    ens.set(G.PSI, psi); ens.set(G.SSTOCH, sig); ens.set_const()
    dts = ens.step(nsteps)
    qs = ens.get(G.Q)
    assert not np.array_equal(qs[0], qs[1])           # different seeds -> different members
    for i in (0, nmem - 1):
        solo = G.Model(G.make_params(**kw), gpu)
        solo.L.msqg_seed_noise(solo.h, 1000 + i)
        solo.set(G.PSI, psi); solo.set(G.SSTOCH, sig); solo.set_const()
        assert [solo.step() for _ in range(nsteps)] == dts[i]
        assert np.array_equal(solo.get(G.Q), qs[i])
    mo = O.Model(O.make_params(**kw))
    mo.set(O.PSI, psi); mo.set(O.SSTOCH, sig); mo.set_const()
    libc.srand(1000 + 1)
    assert [mo.step() for _ in range(nsteps)] == dts[1]
    assert np.array_equal(mo.get(O.Q), qs[1])
    ens.close()
    # production configuration: device noise + red-black smoother; members still equal their solo runs bit for bit
    ens = Ensemble(G.make_params(**kw), nmem, gpu, noise="philox", smoother="rb")
    ens.set(G.PSI, psi); ens.set(G.SSTOCH, sig); ens.set_const()
    dts = ens.step(nsteps)
    qs = ens.get(G.Q)
    assert not np.array_equal(qs[0], qs[1])
    solo = G.Model(G.make_params(**kw), gpu)
    solo.set_smoother("rb")
    solo.L.msqg_seed_noise(solo.h, 1000 + 2); G.check(solo.L.msqg_set_noise_mode(solo.h, 1))
    solo.set(G.PSI, psi); solo.set(G.SSTOCH, sig); solo.set_const()
    assert [solo.step() for _ in range(nsteps)] == dts[2]
    assert np.array_equal(solo.get(G.Q), qs[2])
    ens.close()


@pytest.mark.parametrize("N,nl,nsteps", [(128, 3, 3), (64, 4, 4), (256, 2, 2)])
def test_variable_rossby_number(gpu, N, nl, nsteps):
    """varRo > 0 (msqg/qg.h:1032-1037): Ro, and with it the stretching strl = (Fr/Ro)^2, depends on y; the relax
    kernel then reads per-row Thomas coefficients.  Bit-exact against the oracle, equal cycle counts."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, psi = make_pair(N, nl, varRo=1)
    mo.set_const(); mg.set_const()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()
    so, sg = mo.mgstats(), mg.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    for _ in range(nsteps):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)


@pytest.mark.parametrize("N,nl,varRo,nsteps", [(128, 3, 0, 3), (64, 4, 1, 3), (256, 2, 0, 2)])
def test_stretching_varies_in_x_and_y(gpu, N, nl, varRo, nsteps):
    """Fr from the planetary-geostrophic model (frpg_%dl_N%d.bas -> Frl, msqg/qg.h:957-962): the stretching
    strl = (Fr/Ro)^2 varies with x and y, the relax kernel reads per-CELL Thomas coefficients on every level (built
    from the restricted stretching field, poisson_layer.h:284).  Bit-exact against the oracle, equal cycle counts."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, psi = make_pair(N, nl, varRo=varRo)
    rng = np.random.default_rng(77)
    y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
    fr = np.zeros_like(psi)
    for l in range(nl - 1):
        fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y) + 0.05 * rng.uniform(-1, 1, (N, N)))
    mo.set(O.FR, fr); mg.set(G.FR, fr)
    mo.set_const(); mg.set_const()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))
    z = np.zeros_like(psi)
    mo.set(O.PSI, z); mg.set(G.PSI, z)
    mo.invertq(); mg.invertq()
    so, sg = mo.mgstats(), mg.mgstats()
    assert (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
    assert np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    for _ in range(nsteps):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)
    # the x-dependence matters: the uniform-Fr model gives a different answer
    ref, _, _ = make_pair(N, nl, varRo=varRo)
    ref.set_const()
    for _ in range(nsteps):
        ref.step()
    assert not np.array_equal(ref.get(O.Q), mo.get(O.Q))


@pytest.mark.parametrize("N,nl,ediag,over", [(64, 2, 0, {}), (128, 3, 1, dict(Re=200.)), (64, 4, 0, dict(Re=50., Eks=0.001)),
                                              (64, 3, 0, dict(upg=[0.3, 0.1, 0.], vpg=[0.05, 0., 0.], flsrv=1))])
def test_energy_diagnostics(gpu, N, nl, ediag, over):
    """energy_tend (msqg/qg_energy.h:228-242): advection_de, dissip_de, ekman_friction_de and the running mean
    po_mft accumulated over several steps, bit-exact against the oracle, with viscosity, surface drag and a
    background (planetary-geostrophic) flow."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(N, nl, ediag=ediag, **over)
    mo.set_const(); mg.set_const()
    for k in range(3):
        dto, dtg = mo.step(), mg.step()
        assert dto == dtg
        mo.energy_tend(dto); mg.energy_tend(dtg)
    for fo, fg in ((O.DE_BF, G.DE_BF), (O.DE_VD, G.DE_VD), (O.DE_J1, G.DE_J1), (O.DE_J2, G.DE_J2), (O.DE_J3, G.DE_J3),
                   (O.DE_FT, G.DE_FT), (O.PO_MFT, G.PO_MFT), (O.ZETA, G.ZETA)):
        a, b = mg.get(fg), mo.get(fo)
        assert np.array_equal(a, b), (fg, float(np.abs(a - b).max()))
    assert np.abs(mg.get(G.DE_J1)).max() > 0
    mo.reset_energy(); mg.reset_energy()
    assert not mg.get(G.DE_J1).any() and not mg.get(G.DE_VD).any()


@pytest.mark.parametrize("smoother", ["lex", "rb"])
@pytest.mark.parametrize("N,nl,frfield,over", [(64, 2, 0, {}), (128, 3, 1, dict(Re=200.)), (64, 4, 0, dict(flag_topo=1)),
                                                 (64, 3, 1, dict(upg=[0.3, 0.1, 0.], vpg=[0.05, 0., 0.], flsrv=1, Eks=0.001))])
def test_energy_conserv_variant(gpu, N, nl, frfield, over, smoother):
    """The reference's compile-time variant -DENERGY_CONSERV=1 (msqg/qg.h:310-373, qg_energy.h:33-140) as a runtime
    switch: advection_pv advects the full PV (jacobian(po, qot), ghosts of the evolving list included) and drops
    J(psi_l, psi_l+1); advection_de books jacobian(po, comp_q(po)).  Bit-exact against the oracle: tendency of one
    update_qg, several steps, energy diagnostics -- with uniform and x/y-dependent stretching, a background flow,
    topography, viscosity."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    topo = over.get("flag_topo", 0)
    over = {k: v for k, v in over.items() if k != "flag_topo"}
    mo, mg, psi = make_pair(N, nl, smoother=smoother, **over)
    mo.set_energy_conserv(1); mg.set_energy_conserv(1)
    y, x = np.meshgrid((np.arange(N) + 0.5) / N, (np.arange(N) + 0.5) / N, indexing="ij")
    if frfield:
        fr = np.zeros_like(psi)
        for l in range(nl - 1):
            fr[l] = (0.003 + 0.002 * l) * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y))
        mo.set(O.FR, fr); mg.set(G.FR, fr)
    if topo:
        h = (0.1 * np.exp(-((x - 0.4) ** 2 + (y - 0.6) ** 2) / 0.02))[None]
        mo.set(O.TOPO, h); mg.set(G.TOPO, h)
        mo.L.orc_set_flag_topo(mo.h, 1); G.check(mg.L.msqg_set_flag_topo(mg.h, 1))
    mo.set_const(); mg.set_const()
    assert mg.update(1e10) == mo.update(1e10)
    dqg, dqo = mg.get(G.DQ), mo.get(O.DQ)
    assert np.array_equal(dqg, dqo), float(np.abs(dqg - dqo).max())
    for k in range(3):
        dto, dtg = mo.step(), mg.step()
        assert dto == dtg
        mo.energy_tend(dto); mg.energy_tend(dtg)
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    for fo, fg in ((O.DE_BF, G.DE_BF), (O.DE_VD, G.DE_VD), (O.DE_J1, G.DE_J1), (O.DE_J2, G.DE_J2), (O.DE_J3, G.DE_J3)):
        a, b = mg.get(fg), mo.get(fo)
        assert np.array_equal(a, b), (fg, float(np.abs(a - b).max()))
    # the switch matters: the default build gives different bits
    ref, _, _ = make_pair(N, nl, smoother=smoother, **over)
    if frfield:
        ref.set(O.FR, fr)
    if topo:
        ref.set(O.TOPO, h); ref.L.orc_set_flag_topo(ref.h, 1)
    ref.set_const()
    ref.update(1e10)
    assert not np.array_equal(ref.get(O.DQ), dqo)


@pytest.mark.parametrize("dtflt", [-1.0, 0.05])
def test_pystep_de_python_entry(gpu, dtflt):
    """pystep_de of the SWIG module (msqg/qg_energy.i:30-39) through the ctypes mirror, against the oracle; the
    filter term de_ft (filter_de with pol in the mean slot, qg_energy.h:330) for the default and a positive dtflt"""
    from oracle import oracle as O
    import msom_b200.qg as bas
    N, nl = 64, 3
    kw = base_kw(N, nl, Re=100., dtflt=dtflt, afilt=4.0)
    mo = O.Model(O.make_params(**kw))
    psi = synth_psi(N, nl)
    mo.set(O.PSI, psi); mo.set_const()
    ref = mo.pystep_de(psi)
    import tempfile, os
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "params.in")
        with open(path, "w") as f:
            f.write("#!sh\n")
            for k, v in kw.items():
                f.write("%s = %s\n" % (k, ("[" + ",".join(repr(float(x)) for x in v) + "]") if isinstance(v, (list, tuple)) else repr(v)))
        bas.set_device(gpu)
        bas.read_params(path)
        bas.init_grid(N)
        bas.set_vars()
        bas.set_vars_energy()
        bas.set_const()
        out = [np.zeros_like(psi) for _ in range(6)]
        bas.pystep_de(psi, *out)
        bas.trash_vars_energy()
        bas.trash_vars()
    for a, b in zip(out, ref):
        assert np.array_equal(a, b), float(np.abs(a - b).max())
    assert np.abs(out[5]).max() > 0


@pytest.mark.parametrize("N,nl,nptr,over", [(64, 2, 1, dict(Pe=[40.])), (128, 3, 2, dict(Pe=[50., 0.], ptr_r=[0., 5.])),
                                             (64, 4, 3, dict(Pe=[0., 10., 200.], ptr_r=[2., 0., 0.5]))])
def test_passive_tracers(gpu, N, nl, nptr, over):
    """nptr > 0 (msqg/qg.h:573-588,597-603,634-647): nl*nptr tracers advected by the Arakawa Jacobian, diffused
    (1/Pe) and relaxed (1/ptr_r) with zero-gradient boundaries, stepped with q by the predictor-corrector;
    fused step and plugin sequence, bit-exact against the oracle."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(N, nl, nptr=nptr, **over)
    rng = np.random.default_rng(11)
    tr = rng.standard_normal((nl * nptr, N, N))
    rl = rng.standard_normal((nl * nptr, N, N))
    mo.set(O.PTR, tr); mg.set(G.PTR, tr)
    mo.set(O.PTR_RELAX, rl); mg.set(G.PTR_RELAX, rl)
    mo.set_const(); mg.set_const()
    for _ in range(2):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.PTR), mo.get(O.PTR))
    # plugin surface: update / advance on the evolving and predictor lists
    dt = mg.update(mg.p.DT, G.Q)
    assert dt == mo.update(mo.p.DT)
    assert np.array_equal(mg.get(G.DPTR), mo.get(O.DPTR))
    mg.advance(G.QPRED, G.Q, dt / 2.); mg.update(dt, G.QPRED); mg.advance(G.Q, G.Q, dt)
    mo.L.orc_step.restype  # (oracle: the same iteration through orc_step would redo update; compare via a twin)
    from oracle import oracle as O2
    tw, _, _ = make_pair(N, nl, nptr=nptr, **over)
    tw.set(O2.PTR, tr); tw.set(O2.PTR_RELAX, rl); tw.set_const()
    for _ in range(3):
        tw.step()
    assert np.array_equal(mg.get(G.PTR), tw.get(O2.PTR)) and np.array_equal(mg.get(G.Q), tw.get(O2.Q))
    assert np.isfinite(mg.get(G.PTR)).all() and np.abs(mg.get(G.PTR) - tr).max() > 0


@pytest.mark.parametrize("N,nl,sbc,over", [(64, 2, 0.5, {}), (128, 3, 2.0, dict(Re=300.)), (64, 4, 10.0, dict(upg=[0.2, 0., 0., 0.], flsrv=1))])
def test_partial_slip_boundary(gpu, N, nl, sbc, over):
    """sbc > 0 (msqg/qg.h:185-198): comp_del2 overwrites the vorticity ghosts on the four sides with
    sbc/((0.5*sbc+1)*sq(Delta))*(po[]-po[ghost]); they enter the Jacobians and the viscous terms.
    Bit-exact against the oracle."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    mo, mg, _ = make_pair(N, nl, sbc=sbc, **over)
    mo.set_const(); mg.set_const()
    for _ in range(3):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))
    ref, _, _ = make_pair(N, nl, **over)
    ref.set_const()
    for _ in range(3):
        ref.step()
    assert not np.array_equal(ref.get(O.Q), mo.get(O.Q))      # the boundary condition matters


@pytest.mark.parametrize("N,nl,afilt,modal", [(64, 2, 4.0, 0), (128, 3, 2.5, 0), (64, 4, 7.0, 0), (64, 3, 4.0, 1)])
def test_wavelet_filter(gpu, N, nl, afilt, modal):
    """multi-scale wavelet filter (msqg/qg.h:509-560, SURVEY 8(f) row 3): invertq, [BASILISK] wavelet / sig_lev /
    inverse_wavelet per layer, comp_q and the filter mean, bit-exact against the oracle; then steps continue from
    the filtered state and filter_de (qg_energy.h:207-226) feeds the energy budget."""
    from oracle import oracle as O
    from msom_b200 import capi as G
    if modal and O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev")
    mo, mg, _ = make_pair(N, nl, afilt=afilt, dtflt=0.05, ediag=0, mode_pv_invert=modal)
    mo.set_const(); mg.set_const()
    for _ in range(2):
        assert mg.step() == mo.step()
    mo.wavelet_filter(0.05); mg.wavelet_filter(0.05)
    for fo, fg in ((O.PSI, G.PSI), (O.Q, G.Q), (O.QOF, G.QOF), (O.TMP, G.TMP), (O.SIGLEV, G.SIGLEV)):
        a, b = mg.get(fg), mo.get(fo)
        assert np.array_equal(a, b), (fg, float(np.abs(a - b).max()))
    assert np.abs(mg.get(G.QOF)).max() > 0
    mo.energy_tend(0.01); mg.energy_tend(0.01)
    mo.L.orc_filter_de(mo.h, 0.05); mg.filter_de(0.05)
    for fo, fg in ((O.DE_FT, G.DE_FT), (O.PO_MFT, G.PO_MFT), (O.Q, G.Q), (O.PSI, G.PSI)):
        a, b = mg.get(fg), mo.get(fo)
        assert np.array_equal(a, b), (fg, float(np.abs(a - b).max()))
    assert np.abs(mg.get(G.DE_FT)).max() > 0 and not mg.get(G.PO_MFT).any()
    for _ in range(2):
        assert mg.step() == mo.step()
    assert np.array_equal(mg.get(G.Q), mo.get(O.Q))


@pytest.mark.parametrize("smoother", ["lex", "rb"])
@pytest.mark.parametrize("N,nl", [(128, 3), (256, 4), (32, 2)])
def test_rhs_gather_variant(gpu, N, nl, smoother):
    """MSQG_RHS=gather (L1-gather right-hand side k_rhs instead of the tiled k_rhs_t; the switch is read once per
    process, hence the subprocess) gives the same bits, cycle counts and dt as the oracle, with both sweep orders."""
    import subprocess, sys
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "from common import make_pair\n"
        "from oracle import oracle as O\n"
        "from msom_b200 import capi as G\n"
        "mo, mg, _ = make_pair(%d, %d, smoother=%r)\n"
        "mo.set_const(); mg.set_const()\n"
        "for _ in range(3):\n"
        "    assert mg.step() == mo.step()\n"
        "assert np.array_equal(mg.get(G.Q), mo.get(O.Q)) and np.array_equal(mg.get(G.PSI), mo.get(O.PSI))\n"
        "assert mg.total_cycles == mo.L.orc_total_cycles(mo.h)\n"
        "print('ok')\n") % (ROOT, os.path.join(ROOT, "tests"), N, nl, smoother)
    env = dict(os.environ, MSQG_RHS="gather")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stdout + out.stderr
