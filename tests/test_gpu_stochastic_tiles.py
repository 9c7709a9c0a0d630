"""Stochastic forcing (-D_STOCHASTIC=1, qg_stochastic.h) on the tile machinery: the doubly periodic domain (sbc = -1,
a group of px x py tiles or the 1 x 1 group behind msqg_create) and decomposed closed-basin groups.

The noise is pointwise, so a tile draws only its own cells: the Philox counter is the global cell-layer index, and the
libc replay runs through the whole N^2 x nl rand() stream of the undecomposed grid on every tile and keeps its window.
So a group gives the bits of the undecomposed model and, with libc noise, of the oracle drawing from the process-wide
rand() after srand(seed)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from common import base_kw, periodic_psi, rel_l2, synth_psi

pytestmark = pytest.mark.gpu
libc = C.CDLL(None)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STOCH = dict(stochastic=1, tr_stoch=10., amp_stoch=1.)


def _sigma(N, nl):
    """noise amplitude varying by layer, as in test_stochastic_forcing_philox"""
    return np.full((nl, N, N), 1e-3) * (1 + np.arange(nl)[:, None, None])


def _oracle(kw, psi, sig, decomp=None):
    from oracle import oracle as O
    mo = O.Model(O.make_params(**kw))
    if decomp:
        mo.L.orc_set_decomp(mo.h, *decomp)
    else:
        mo.set_smoother("rb")
    mo.set(O.PSI, psi); mo.set(O.SSTOCH, sig); mo.set_const()
    return mo


def _group(kw, px, py, agg_n, gpu, psi, sig, seed, mode="libc", smoother="rb"):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    g = Group(G.make_params(**kw), px, py, agg_n, gpu, smoother=smoother, noise=mode, seed=seed)
    g.set_global(G.PSI, psi); g.set_global(G.SSTOCH, sig); g.set_const()
    return g


def _model(kw, gpu, psi, sig, seed, mode="libc", smoother="rb"):
    from msom_b200 import capi as G
    m = G.Model(G.make_params(**kw), gpu)
    if kw.get("sbc", 0) != -1:
        m.set_smoother(smoother)
    m.L.msqg_seed_noise(m.h, seed); G.check(m.L.msqg_set_noise_mode(m.h, {"libc": 0, "philox": 1}[mode]))
    m.set(G.PSI, psi); m.set(G.SSTOCH, sig); m.set_const()
    return m


def _oracle_steps(mo, nsteps, seed):
    libc.srand(seed)                       # the oracle draws from the process-wide rand() like the reference
    return [mo.step() for _ in range(nsteps)]


@pytest.mark.parametrize("N,nl,px,py", [(64, 3, 1, 1), (128, 2, 2, 1), (128, 4, 2, 2), (128, 3, 1, 2), (64, 10, 1, 1)])
def test_periodic_stochastic_libc_matches_oracle(gpu, N, nl, px, py):
    from oracle import oracle as O
    from msom_b200 import capi as G
    seed, nsteps = 321, 4
    kw = base_kw(N, nl, sbc=-1., **STOCH)
    psi, sig = periodic_psi(N, nl), _sigma(N, nl)
    mo = _oracle(kw, psi, sig)
    dto = _oracle_steps(mo, nsteps, seed)
    g = _group(kw, px, py, 0, gpu, psi, sig, seed)
    assert [g.step() for _ in range(nsteps)] == dto
    assert g.total_cycles == mo.L.orc_total_cycles(mo.h)
    for fg, fo in ((G.NSTOCH, O.NSTOCH), (G.Q, O.Q), (G.PSI, O.PSI)):
        assert np.array_equal(g.get_global(fg), mo.get(fo)), fg
    assert np.abs(mo.get(O.NSTOCH)).max() > 0
    g.close()


def test_periodic_stochastic_philox(gpu):
    """device noise: 2 x 1 and 2 x 2 periodic groups give the bits of the 1 x 1 periodic handle; against the oracle's
    restatement of the generator with the tolerances of test_stochastic_forcing_philox (CUDA and glibc log/cos may
    differ in the last place)"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    N, nl, nsteps, seed = 128, 3, 4, 4242
    kw = base_kw(N, nl, sbc=-1., **STOCH)
    psi, sig = periodic_psi(N, nl), _sigma(N, nl)
    one = _model(kw, gpu, psi, sig, seed, "philox")
    dts = [one.step() for _ in range(nsteps)]
    ref = {f: one.get(f) for f in (G.NSTOCH, G.Q, G.PSI)}
    for px, py in ((2, 1), (2, 2)):
        g = _group(kw, px, py, 0, gpu, psi, sig, seed, "philox")
        assert [g.step() for _ in range(nsteps)] == dts
        assert g.total_cycles == one.total_cycles
        for f, a in ref.items():
            assert np.array_equal(g.get_global(f), a), (px, py, f)
        g.close()
    mo = _oracle(kw, psi, sig)
    mo.L.orc_set_noise_mode(mo.h, 1, seed)
    for dt in dts:
        assert abs(dt - mo.step()) <= 1e-15
    a, b = ref[G.NSTOCH], mo.get(O.NSTOCH)
    assert np.abs(a - b).max() <= 1e-13 * np.abs(b).max() and np.abs(b).max() > 0
    for fg, fo in ((G.Q, O.Q), (G.PSI, O.PSI)):
        assert rel_l2(ref[fg], mo.get(fo)) <= 1e-10


@pytest.mark.parametrize("p2p", [1, 0])
@pytest.mark.parametrize("N,nl,px,py", [(128, 3, 2, 1), (256, 2, 2, 2), (256, 4, 4, 2), (256, 3, 1, 2)])
def test_red_black_group_stochastic(gpu, N, nl, px, py, p2p, monkeypatch):
    """closed basin: a red-black group with libc noise gives the bits of the undecomposed red-black model and of the
    oracle; with Philox noise the bits of the undecomposed model"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    monkeypatch.setenv("MSQG_P2P", str(p2p))
    agg_n = 128 if px == 4 else 64        # as test_red_black_group_equals_single_gpu_and_oracle
    seed, nsteps = 77, 3
    kw = base_kw(N, nl, **STOCH)
    psi, sig = synth_psi(N, nl), _sigma(N, nl)
    mo = _oracle(kw, psi, sig)
    dto = _oracle_steps(mo, nsteps, seed)
    for mode in ("libc", "philox"):
        s = _model(kw, gpu, psi, sig, seed, mode)
        g = _group(kw, px, py, agg_n, gpu, psi, sig, seed, mode)
        assert g.transport == ("peer-memory" if p2p else "nccl")
        dts = [g.step() for _ in range(nsteps)]
        assert dts == [s.step() for _ in range(nsteps)]
        assert g.total_cycles == s.total_cycles
        for f in (G.NSTOCH, G.Q, G.PSI):
            assert np.array_equal(g.get_global(f), s.get(f)), (mode, f)
        if mode == "libc":
            assert dts == dto and g.total_cycles == mo.L.orc_total_cycles(mo.h)
            for fg, fo in ((G.NSTOCH, O.NSTOCH), (G.Q, O.Q), (G.PSI, O.PSI)):
                assert np.array_equal(g.get_global(fg), mo.get(fo)), fg
        g.close(); s.close()


def test_red_black_group_stochastic_modal(gpu):
    """the vertical-mode inversion (mode_pv_invert = 1) under stochastic forcing on a red-black group, libc noise"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    if O._lapack_path() is None:
        pytest.skip("no LAPACK dgeev (eigmode.h:153)")
    N, nl, px, py, seed, nsteps = 128, 3, 2, 1, 5, 3
    kw = base_kw(N, nl, mode_pv_invert=1, **STOCH)
    psi, sig = synth_psi(N, nl), _sigma(N, nl)
    mo = _oracle(kw, psi, sig)
    dto = _oracle_steps(mo, nsteps, seed)
    s = _model(kw, gpu, psi, sig, seed)
    g = _group(kw, px, py, 64, gpu, psi, sig, seed)
    assert [g.step() for _ in range(nsteps)] == [s.step() for _ in range(nsteps)] == dto
    for fg, fo in ((G.NSTOCH, O.NSTOCH), (G.Q, O.Q), (G.PSI, O.PSI)):
        assert np.array_equal(g.get_global(fg), s.get(fg)), fg
        assert np.array_equal(g.get_global(fg), mo.get(fo)), fg


def test_lexicographic_group_stochastic_matches_oracle_decomposition(gpu):
    """the lexicographic (block Gauss-Seidel) group with libc noise against the oracle's emulation of the same
    decomposition (orc_set_decomp), as scripts/dist_check.py lex"""
    from oracle import oracle as O
    from msom_b200 import capi as G
    N, nl, px, py, agg_n, seed, nsteps = 128, 3, 2, 2, 32, 9, 3
    kw = base_kw(N, nl, **STOCH)
    psi, sig = synth_psi(N, nl), _sigma(N, nl)
    mo = _oracle(kw, psi, sig, decomp=(px, py, agg_n))
    dto = _oracle_steps(mo, nsteps, seed)
    g = _group(kw, px, py, agg_n, gpu, psi, sig, seed, smoother="lex")
    assert [g.step() for _ in range(nsteps)] == dto
    assert g.total_cycles == mo.L.orc_total_cycles(mo.h)
    for fg, fo in ((G.NSTOCH, O.NSTOCH), (G.Q, O.Q), (G.PSI, O.PSI)):
        assert np.array_equal(g.get_global(fg), mo.get(fo)), fg


@pytest.mark.parametrize("mode", ["libc", "philox"])
def test_periodic_stochastic_plugin_sequence_equals_fused_step(gpu, mode):
    """update_qg / advance_qg on the periodic handle, called as the predictor-corrector does, draw the noise at the
    same stages as the fused step and give its bits"""
    from msom_b200 import capi as G
    N, nl, seed = 64, 3, 11
    kw = base_kw(N, nl, sbc=-1., **STOCH)
    psi, sig = periodic_psi(N, nl), _sigma(N, nl)
    a, b = _model(kw, gpu, psi, sig, seed, mode), _model(kw, gpu, psi, sig, seed, mode)
    for _ in range(3):
        dt = a.update(a.p.DT, G.Q)
        a.advance(G.QPRED, G.Q, dt / 2.)
        a.update(dt, G.QPRED)
        a.advance(G.Q, G.Q, dt)
        assert b.step() == dt
    for f in (G.NSTOCH, G.Q, G.PSI):
        assert np.array_equal(a.get(f), b.get(f)), f
    assert np.abs(a.get(G.NSTOCH)).max() > 0


def test_periodic_stochastic_ensemble(gpu):
    """periodic members (each a 1 x 1 periodic group) with device noise: members differ, each equals its solo run;
    periodic members need the red-black smoother"""
    from msom_b200 import capi as G
    from msom_b200.ensemble import Ensemble
    N, nl, nmem, nsteps = 64, 3, 3, 3
    kw = base_kw(N, nl, sbc=-1., **STOCH)
    psi, sig = periodic_psi(N, nl), _sigma(N, nl)
    ens = Ensemble(G.make_params(**kw), nmem, gpu, noise="philox", smoother="rb")
    ens.set(G.PSI, psi); ens.set(G.SSTOCH, sig); ens.set_const()
    dts = ens.step(nsteps)
    qs = ens.get(G.Q)
    assert not np.array_equal(qs[0], qs[1]) and not np.array_equal(qs[1], qs[2])
    for i in range(nmem):
        solo = _model(kw, gpu, psi, sig, 1000 + i, "philox")
        assert [solo.step() for _ in range(nsteps)] == dts[i]
        assert np.array_equal(solo.get(G.Q), qs[i]) and np.array_equal(solo.get(G.PSI), ens.get(G.PSI)[i])
        solo.close()
    ens.close()
    with pytest.raises(G.MsqgError):
        Ensemble(G.make_params(**kw), 2, gpu, noise="philox", smoother="lex")


def test_qg_exe_periodic_stochastic(gpu, tmp_path):
    """./qg.e --stochastic with sbc = -1 and s_stoch_3l_N64.bas: po/qo files byte for byte those of the oracle's run()
    after srand(1) (the rand() state a reference process starts from)"""
    from oracle import oracle as O
    from test_gpu_host import _write_params
    N, nl = 64, 3
    wd = tmp_path / "gpu"; wd.mkdir()
    wo = tmp_path / "orc"; wo.mkdir()
    _write_params(str(wd / "params.in"), N, nl, tend=0.1, dtout=0.05, extra="sbc = -1\ntr_stoch = 10.\namp_stoch = 1.\n")
    psi, sig = periodic_psi(N, nl), _sigma(N, nl)
    O.lib().orc_write_bas(str(wd / "p0.bas").encode(), nl, N, 80., psi)
    O.lib().orc_write_bas(str(wd / ("s_stoch_%dl_N%d.bas" % (nl, N))).encode(), nl, N, 80., sig)
    exe = os.path.join(ROOT, "msom_b200", "lib", "qg.e")
    out = subprocess.run([exe, "--stochastic"], cwd=str(wd), capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "s_stoch_3l_N64.bas .. ok" in out.stdout
    po = O.Params(); O.lib().orc_default_params(po); O.lib().orc_read_params(str(wd / "params.in").encode(), po)
    po.stochastic = 1
    assert po.sbc == -1 and po.itr_stoch == 0.1
    mo = O.Model(po); mo.set_smoother("rb")
    p0 = np.zeros_like(psi); O.lib().orc_read_bas(str(wd / "p0.bas").encode(), nl, N, 80., p0)
    s0 = np.zeros_like(sig); O.lib().orc_read_bas(str(wd / ("s_stoch_%dl_N%d.bas" % (nl, N))).encode(), nl, N, 80., s0)
    mo.set(O.PSI, p0); mo.L.orc_remove_mean_psi(mo.h); mo.set(O.SSTOCH, s0); mo.set_const()
    libc.srand(1)
    assert mo.run(outdir=str(wo)) > 0
    gdir = wd / "outdir_0001"
    names = sorted(f for f in os.listdir(wo) if f.endswith(".bas"))
    assert len(names) == 6
    for f in names:
        assert (gdir / f).read_bytes() == (wo / f).read_bytes(), f


def test_stochastic_refusals_that_stay(gpu):
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    with pytest.raises(G.MsqgError):     # the vertical-mode inversion is not built for periodic boundaries
        G.Model(G.make_params(**base_kw(64, 2, sbc=-1., mode_pv_invert=1, **STOCH)), gpu)
    for sbc in (0., -1.):                # tracers are not advanced by the stochastic advance_qg (qg_stochastic.h:139-147)
        with pytest.raises(G.MsqgError):
            G.Model(G.make_params(**base_kw(64, 2, sbc=sbc, nptr=1, **STOCH)), gpu)
    # a Python group with stochastic forcing is told its noise stream when it is built, for every tile at once
    N, nl = 128, 2
    kw = base_kw(N, nl, **STOCH)
    psi, sig = synth_psi(N, nl), _sigma(N, nl)
    for smoother in ("rb", "lex"):
        with pytest.raises(G.MsqgError, match="stochastic") as e:
            Group(G.make_params(**kw), 2, 1, 64, gpu, smoother=smoother)
        assert e.value.code == G.ERR_ARG
        Group(G.make_params(**kw), 2, 1, 64, gpu, smoother=smoother, noise="philox", seed=3).close()
    # tiles of one group seeded differently would each draw a different field: refused at the step
    g = _group(kw, 2, 1, 64, gpu, psi, sig, 5)
    g.L.msqg_seed_noise(g.L.msqg_group_tile(g.h, 1), 6)
    with pytest.raises(G.MsqgError, match="seed"):
        g.step()
    g.seed_noise(5)                      # seeded alike again: the group steps
    assert g.step() > 0
    g.L.msqg_set_noise_mode(g.L.msqg_group_tile(g.h, 0), 1)
    with pytest.raises(G.MsqgError, match="mode"):
        g.step()
    g.close()


def test_nccl_stochastic_two_gpus(gpu):
    """the NCCL back-end with libc noise, closed basin and periodic, bit for bit against the oracle (torchrun on 2
    GPUs); skipped on a single-GPU box"""
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    for mode in ("rbstoch", "rbperstoch"):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", "29536", os.path.join(ROOT, "scripts", "dist_check.py"), mode],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "DIST_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
