"""ctypes binding of the CPU oracle (oracle/msqg_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package
(msom_b200) must never import this module.
"""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
MAXL = 32

PSI, Q, PSIPG, FR, QFORC, TOPO, RD, SSTOCH, ZETA, DQ, STR, NSTOCH, IBU, CL2M, CM2L, PM, QM, TMP, ZETAP = range(19)
DE_BF, DE_VD, DE_J1, DE_J2, DE_J3, DE_FT, PO_MFT = range(19, 26)  # energy diagnostics, qg_energy.h
PTR, PTR_RELAX, DPTR = range(26, 29)  # passive tracers, qg.h:100-101
QOF, SIGLEV = 29, 30  # wavelet filter: filter mean qofl (qg.h:27), sig_lev (qg.h:49)


class Params(C.Structure):
    _fields_ = (
        [(k, C.c_int) for k in ("N", "nl", "ediag", "varRo", "nptr", "flsrv")]
        + [(k, C.c_double) for k in ("L0", "Rom", "Ekb", "Eks", "tau0", "Re", "Re4", "sbc", "beta",
                                     "afilt", "Lfmax", "DT", "tend", "dtout", "dtflt", "CFL")]
        + [(k, C.c_double * MAXL) for k in ("Fr", "dh", "upg", "vpg")]
        + [("iRe", C.c_double), ("iRe4", C.c_double), ("stochastic", C.c_int),
           ("tr_stoch", C.c_double), ("itr_stoch", C.c_double), ("amp_stoch", C.c_double),
           ("mode_pv_invert", C.c_int)]
        + [(k, C.c_double * MAXL) for k in ("ptr_r", "Pe", "ptr_ir", "iPe")]
        + [("px", C.c_int), ("py", C.c_int)]
    )


class MgStats(C.Structure):
    _fields_ = [("i", C.c_int), ("resb", C.c_double), ("resa", C.c_double), ("sum", C.c_double),
                ("nrelax", C.c_int)]


def build(force=False):
    out = os.path.join(_HERE, "build")
    libs = [os.path.join(out, "libmsqg_oracle.so"), os.path.join(out, "libmsqg_oracle_omp.so")]
    src = os.path.join(_HERE, "msqg_oracle.c")
    stale = force or any((not os.path.exists(l)) or os.path.getmtime(l) < os.path.getmtime(src) for l in libs)
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "-s"], stdout=subprocess.DEVNULL)
    return libs


def _lapack_path():
    try:
        import scipy
        c = glob.glob(os.path.join(os.path.dirname(scipy.__file__), "..", "scipy.libs", "libscipy_openblas*.so"))
        if c:
            return os.path.abspath(c[0])
    except Exception:
        pass
    return None


_libs = {}


def lib(omp=False):
    key = "omp" if omp else "serial"
    if key in _libs:
        return _libs[key]
    paths = build()
    lp = _lapack_path()
    if lp and "MSQG_ORACLE_LAPACK" not in os.environ:
        os.environ["MSQG_ORACLE_LAPACK"] = lp
    L = C.CDLL(paths[1] if omp else paths[0])
    dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    vp = C.c_void_p
    L.orc_default_params.argtypes = [C.POINTER(Params)]
    L.orc_read_params.argtypes = [C.c_char_p, C.POINTER(Params)]
    L.orc_read_params.restype = C.c_int
    L.orc_create.argtypes = [C.POINTER(Params)]
    L.orc_create.restype = vp
    L.orc_destroy.argtypes = [vp]
    L.orc_nfields.argtypes = [vp, C.c_int]
    L.orc_nfields.restype = C.c_int
    L.orc_set_field.argtypes = [vp, C.c_int, dp]
    L.orc_get_field.argtypes = [vp, C.c_int, dp]
    L.orc_set_const.argtypes = [vp]
    L.orc_set_const.restype = C.c_int
    L.orc_set_flag_topo.argtypes = [vp, C.c_int]
    L.orc_set_decomp.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.orc_set_smoother.argtypes = [vp, C.c_int]
    L.orc_set_energy_conserv.argtypes = [vp, C.c_int]
    L.orc_set_noise_mode.argtypes = [vp, C.c_int, C.c_uint]
    L.orc_get_smoother.argtypes = [vp]
    L.orc_get_smoother.restype = C.c_int
    L.orc_init_noise.argtypes = [vp, C.c_uint]
    L.orc_remove_mean_psi.argtypes = [vp]
    L.orc_invertq.argtypes = [vp]
    L.orc_comp_q.argtypes = [vp]
    L.orc_last_mgstats.argtypes = [vp, C.c_int]
    L.orc_last_mgstats.restype = MgStats
    L.orc_total_cycles.argtypes = [vp]
    L.orc_total_cycles.restype = C.c_int
    L.orc_test_cycles.argtypes = [vp, C.c_int, np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS"), C.c_int, dp]
    L.orc_test_cycles.restype = C.c_int
    L.orc_update.argtypes = [vp, C.c_double]
    L.orc_update.restype = C.c_double
    L.orc_step.argtypes = [vp]
    L.orc_step.restype = C.c_double
    L.orc_run.argtypes = [vp, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.orc_run.restype = C.c_int
    L.orc_time.argtypes = [vp]
    L.orc_time.restype = C.c_double
    L.orc_ke1.argtypes = [vp]
    L.orc_ke1.restype = C.c_double
    L.orc_pystep_bfn.argtypes = [vp, dp, dp, C.c_double, C.c_int]
    L.orc_wavelet_filter.argtypes = [vp, C.c_double]
    L.orc_get_siglev.argtypes = [vp, C.c_int, dp]
    L.orc_filter_de.argtypes = [vp, C.c_double]
    L.orc_energy_tend.argtypes = [vp, C.c_double]
    L.orc_reset_energy.argtypes = [vp]
    L.orc_pystep_de.argtypes = [vp, dp, dp, dp, dp, dp, dp, dp, C.c_int]
    L.orc_pyq2p.argtypes = [vp, dp, dp]
    L.orc_pyp2q.argtypes = [vp, dp, dp]
    L.orc_test_relax.argtypes = [C.c_int, C.c_int, C.c_double, dp, dp, dp, dp, C.c_int, C.c_int, C.c_int]
    L.orc_test_relax_rb.argtypes = [C.c_int, C.c_int, C.c_double, dp, dp, dp, dp, C.c_int]
    L.orc_test_relax_scalar_rb.argtypes = [C.c_int, C.c_double, dp, dp, dp, C.c_int]
    L.orc_test_residual.argtypes = [C.c_int, C.c_int, C.c_double, dp, dp, dp, dp, dp]
    L.orc_test_residual.restype = C.c_double
    L.orc_test_restrict.argtypes = [C.c_int, C.c_int, dp, dp]
    L.orc_test_prolong.argtypes = [C.c_int, C.c_int, dp, dp]
    L.orc_test_relax_scalar.argtypes = [C.c_int, C.c_double, dp, dp, dp, C.c_int]
    L.orc_test_residual_scalar.argtypes = [C.c_int, C.c_double, dp, dp, dp, dp]
    L.orc_test_residual_scalar.restype = C.c_double
    L.orc_eigmod_column.argtypes = [C.c_int, dp, dp, C.c_double, dp, dp, dp]
    L.orc_eigmod_column.restype = C.c_int
    L.orc_write_bas.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_double, dp]
    L.orc_write_bas.restype = C.c_int
    L.orc_read_bas.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_double, dp]
    L.orc_read_bas.restype = C.c_int
    _libs[key] = L
    return L


def make_params(omp=False, **kw):
    """Params with reference defaults, overridden by kw; applies the derived
    quantities of read_params (qg.h:739-746) exactly like the file path does."""
    L = lib(omp)
    p = Params()
    L.orc_default_params(C.byref(p))
    for k, v in kw.items():
        if k in ("Fr", "dh", "upg", "vpg", "ptr_r", "Pe"):
            arr = getattr(p, k)
            for i, x in enumerate(v):
                arr[i] = float(x)
        else:
            setattr(p, k, v)
    if p.Re != 0:
        p.iRe = 1 / p.Re
        p.DT = 0.5 * min(p.DT, (p.L0 / p.N) ** 2 * p.Re / 4.0)
    if p.Re4 != 0:
        p.iRe4 = -1 / p.Re4
        d2 = (p.L0 / p.N) * (p.L0 / p.N)
        p.DT = 0.5 * min(p.DT, d2 * d2 * p.Re4 / 32.0)
    if p.tr_stoch != 0:
        p.itr_stoch = 1 / p.tr_stoch
    for nt in range(p.nptr):  # qg.h:751-754
        p.ptr_ir[nt] = 0.0 if p.ptr_r[nt] == 0 else 1 / p.ptr_r[nt]
        p.iPe[nt] = 0.0 if p.Pe[nt] == 0 else 1 / p.Pe[nt]
    return p


class Model:
    """Thin object wrapper mirroring the reference call order
    read_params -> init_grid -> set_vars -> set_const -> (...)."""

    def __init__(self, params, omp=False):
        self.L = lib(omp)
        self.p = params
        self.N, self.nl = params.N, params.nl
        self.h = self.L.orc_create(C.byref(params))

    def close(self):
        if self.h:
            self.L.orc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def nfields(self, fid):
        return self.L.orc_nfields(self.h, fid)

    def set(self, fid, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float64)
        assert arr.shape == (self.nfields(fid), self.N, self.N), (arr.shape, self.nfields(fid))
        self.L.orc_set_field(self.h, fid, arr)

    def get(self, fid):
        out = np.zeros((self.nfields(fid), self.N, self.N))
        self.L.orc_get_field(self.h, fid, out)
        return out

    def set_smoother(self, name):
        """'lex' (reference order, default) or 'rb' (red-black ordering of the same cell update)"""
        self.L.orc_set_smoother(self.h, {"lex": 0, "rb": 1}[name])

    def set_energy_conserv(self, on):
        """the reference's -DENERGY_CONSERV=1 build (qg.h:310-373) as a runtime switch"""
        self.L.orc_set_energy_conserv(self.h, int(bool(on)))

    def set_const(self):
        rc = self.L.orc_set_const(self.h)
        if rc:
            raise RuntimeError("orc_set_const failed rc=%d" % rc)

    def invertq(self):
        self.L.orc_invertq(self.h)

    def comp_q(self):
        self.L.orc_comp_q(self.h)

    def mgstats(self, mode=-1):
        return self.L.orc_last_mgstats(self.h, mode)

    def test_cycles(self, nrelax, mode=-1):
        """len(nrelax) multigrid cycles, cycle k with nrelax[k] sweeps per level (orc_test_cycles): the unknown (PSI, or
        plane `mode` of PM) is updated in place; returns the residual max norm after every cycle"""
        sched = np.ascontiguousarray(nrelax, dtype=np.int32)
        resa = np.zeros(len(sched))
        if self.L.orc_test_cycles(self.h, mode, sched, len(sched), resa):
            raise ValueError("orc_test_cycles refused mode %d / schedule %s" % (mode, list(sched)))
        return resa

    def update(self, dtmax):
        return self.L.orc_update(self.h, dtmax)

    def step(self):
        return self.L.orc_step(self.h)

    def run(self, max_steps=-1, outdir=None, verbose=0):
        return self.L.orc_run(self.h, max_steps, 1 if outdir else 0, (outdir or "").encode(), verbose)

    @property
    def t(self):
        return self.L.orc_time(self.h)

    def ke1(self):
        return self.L.orc_ke1(self.h)

    def wavelet_filter(self, dtflt):
        self.L.orc_wavelet_filter(self.h, dtflt)

    def siglev(self, level):
        n = 1 << level
        out = np.zeros((n, n))
        self.L.orc_get_siglev(self.h, level, out)
        return out

    def energy_tend(self, dt):
        self.L.orc_energy_tend(self.h, dt)

    def reset_energy(self):
        self.L.orc_reset_energy(self.h)

    def pystep_de(self, po, onlyKE=0):
        out = [np.zeros_like(po) for _ in range(6)]
        self.L.orc_pystep_de(self.h, np.ascontiguousarray(po), *out, onlyKE)
        return out
