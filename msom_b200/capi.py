"""ctypes binding of the handle-based C ABI (include/msqg.h, layer 1).

Thin marshaling only: numpy float64 C-contiguous arrays [layer][y][x] in, the
same out.  All compute happens in libmsqg_cuda.so (hand-written sm_100a
kernels); there is no CPU path and loading fails loudly if the library is
missing.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_CUDA = os.path.join(_HERE, "lib", "libmsqg_cuda.so")
MAXL = 32

(PSI, Q, PSIPG, FR, QFORC, TOPO, RD, SSTOCH, ZETA, DQ, STR, NSTOCH, IBU, CL2M, CM2L, PM, QM, TMP, ZETAP,
 QPRED, SIGFILT, DE_BF, DE_VD, DE_J1, DE_J2, DE_J3, DE_FT, PO_MFT, PTR, PTR_RELAX, DPTR, QOF, SIGLEV) = range(33)

OK, ERR_ARG, ERR_CUDA, ERR_FILE, ERR_CONFIG, ERR_NOCONV = 0, -1, -2, -3, -4, -5


class Params(C.Structure):
    """msqg_params (keys of params.in, msqg/qg.h:698-731, + derived values)."""
    _fields_ = (
        [(k, C.c_int) for k in ("N", "nl", "ediag", "varRo", "nptr", "flsrv")]
        + [(k, C.c_double) for k in ("L0", "Rom", "Ekb", "Eks", "tau0", "Re", "Re4", "sbc", "beta",
                                     "afilt", "Lfmax", "DT", "tend", "dtout", "dtflt", "CFL")]
        + [(k, C.c_double * MAXL) for k in ("Fr", "dh", "upg", "vpg")]
        + [("iRe", C.c_double), ("iRe4", C.c_double), ("stochastic", C.c_int),
           ("tr_stoch", C.c_double), ("itr_stoch", C.c_double), ("amp_stoch", C.c_double),
           ("mode_pv_invert", C.c_int)]
        + [(k, C.c_double * MAXL) for k in ("ptr_r", "Pe", "ptr_ir", "iPe")]
    )


class MgStats(C.Structure):
    _fields_ = [("i", C.c_int), ("resb", C.c_double), ("resa", C.c_double), ("sum", C.c_double),
                ("nrelax", C.c_int)]


class MsqgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("msqg error %d: %s" % (code, msg))
        self.code = code


_lib = None


def _find_lapack():
    """eigmod (msqg/eigmode.h:153) needs LAPACK dgeev; point the library at one."""
    if "MSQG_LAPACK" in os.environ:
        return
    import glob
    try:
        import scipy
        c = glob.glob(os.path.join(os.path.dirname(scipy.__file__), "..", "scipy.libs", "libscipy_openblas*.so"))
        if c:
            os.environ["MSQG_LAPACK"] = os.path.abspath(c[0])
    except Exception:
        pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_CUDA):
        raise ImportError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the msqg timestep has no CPU fallback)" % LIB_CUDA)
    _find_lapack()
    L = C.CDLL(LIB_CUDA, mode=C.RTLD_GLOBAL)
    dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    vp = C.c_void_p
    pd = C.POINTER(C.c_double)
    L.msqg_last_error.restype = C.c_char_p
    L.msqg_default_params.argtypes = [C.POINTER(Params)]
    L.msqg_derive_params.argtypes = [C.POINTER(Params)]
    L.msqg_read_params.argtypes = [C.c_char_p, C.POINTER(Params)]
    L.msqg_create.argtypes = [C.POINTER(Params), C.c_int, C.POINTER(vp)]
    L.msqg_destroy.argtypes = [vp]
    L.msqg_set_stream.argtypes = [vp, vp]
    L.msqg_nfields.argtypes = [vp, C.c_int]
    L.msqg_energy_tend.argtypes = [vp, C.c_double, C.c_double]
    L.msqg_wavelet_filter.argtypes = [vp, C.c_double]
    L.msqg_invert_filter_mean.argtypes = [vp]
    L.msqg_filter_de.argtypes = [vp, C.c_double, C.c_double]
    L.msqg_filter_de_pm.argtypes = [vp, C.c_double, C.c_double, C.c_int]
    L.msqg_reset_energy.argtypes = [vp]
    L.msqg_set_field.argtypes = [vp, C.c_int, dp]
    L.msqg_get_field.argtypes = [vp, C.c_int, dp]
    L.msqg_set_flag_topo.argtypes = [vp, C.c_int]
    L.msqg_set_smoother.argtypes = [vp, C.c_int]
    L.msqg_get_smoother.argtypes = [vp]
    L.msqg_set_energy_conserv.argtypes = [vp, C.c_int]
    L.msqg_ensemble_create.argtypes = [C.POINTER(Params), C.c_int, C.c_int, C.POINTER(C.c_uint), C.c_int, C.c_int, C.POINTER(vp)]
    L.msqg_ensemble_destroy.argtypes = [vp]
    L.msqg_ensemble_destroy.restype = None
    L.msqg_ensemble_size.argtypes = [vp]
    L.msqg_ensemble_member.argtypes = [vp, C.c_int]
    L.msqg_ensemble_member.restype = vp
    L.msqg_ensemble_set_const.argtypes = [vp]
    L.msqg_ensemble_step.argtypes = [vp, C.c_int, pd]
    L.msqg_ensemble_time.argtypes = [vp, C.c_int]
    L.msqg_ensemble_time.restype = C.c_double
    L.msqg_set_field_async.argtypes = [vp, C.c_int, dp]
    L.msqg_set_field_commit.argtypes = [vp]
    L.msqg_get_field_async.argtypes = [vp, C.c_int, dp]
    L.msqg_io_wait.argtypes = [vp]
    L.msqg_get_energy_conserv.argtypes = [vp]
    L.msqg_set_keep_dq.argtypes = [vp, C.c_int]
    L.msqg_set_dissipation.argtypes = [vp, C.c_double, C.c_double, C.c_double, C.c_double]
    L.msqg_set_const.argtypes = [vp]
    L.msqg_invertq.argtypes = [vp, C.c_int]
    L.msqg_comp_q.argtypes = [vp]
    L.msqg_last_mgstats.argtypes = [vp, C.c_int, C.POINTER(MgStats)]
    L.msqg_total_cycles.argtypes = [vp]
    L.msqg_total_cycles.restype = C.c_long
    L.msqg_update.argtypes = [vp, C.c_int, C.c_double, pd]
    L.msqg_advance.argtypes = [vp, C.c_int, C.c_int, C.c_double]
    L.msqg_step.argtypes = [vp, C.c_double, C.c_double, pd, pd]
    L.msqg_ke1.argtypes = [vp, pd]
    L.msqg_tendency_bfn.argtypes = [vp, C.c_double]
    L.msqg_get_ts_previous.argtypes = [vp]
    L.msqg_get_ts_previous.restype = C.c_double
    L.msqg_set_ts_previous.argtypes = [vp, C.c_double]
    L.msqg_seed_noise.argtypes = [vp, C.c_uint]
    L.msqg_set_noise_mode.argtypes = [vp, C.c_int]
    L.msqg_launch_count.argtypes = [vp]
    L.msqg_launch_count.restype = C.c_long
    L.msqg_test_relax.argtypes = [vp, C.c_int, dp, dp, C.c_int]
    L.msqg_test_relax_scalar.argtypes = [vp, C.c_int, C.c_double, dp, dp, C.c_int]
    L.msqg_test_residual.argtypes = [vp, dp, dp, dp, pd]
    L.msqg_test_residual_levels.argtypes = [vp, C.c_int, dp, dp, dp, pd, C.POINTER(C.c_int)]
    L.msqg_test_cycles.argtypes = [vp, C.c_int, np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS"), C.c_int, dp]
    L.msqg_test_restrict.argtypes = [vp, C.c_int, dp, dp]
    L.msqg_test_prolong.argtypes = [vp, C.c_int, dp, dp]
    L.msqg_test_div.argtypes = [C.c_int, dp, dp, dp, dp, C.c_int]
    L.msqg_time_vcycle.argtypes = [vp, C.c_int, C.c_int, pd]
    L.msqg_profile_enable.argtypes = [vp, C.c_int]
    L.msqg_profile_read.argtypes = [vp, pd, C.POINTER(C.c_long), C.POINTER(C.c_long)]
    L.msqg_reset_field.argtypes = [vp, C.c_int]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise MsqgError(rc, lib().msqg_last_error().decode(errors="replace"))


def make_params(**kw):
    """msqg_params with the reference defaults, overridden by kw, then the
    derived values of read_params (msqg/qg.h:739-746)."""
    p = Params()
    lib().msqg_default_params(C.byref(p))
    for k, v in kw.items():
        if k in ("Fr", "dh", "upg", "vpg", "ptr_r", "Pe"):
            arr = getattr(p, k)
            for i, x in enumerate(v):
                arr[i] = float(x)
        else:
            setattr(p, k, v)
    lib().msqg_derive_params(C.byref(p))
    return p


def read_params(path, stochastic=0, mode_pv_invert=0):
    p = Params()
    lib().msqg_default_params(C.byref(p))
    p.stochastic = stochastic
    p.mode_pv_invert = mode_pv_invert
    check(lib().msqg_read_params(str(path).encode(), C.byref(p)))
    return p


class Model:
    """One msqg model resident on one GPU (msqg_create .. msqg_destroy)."""

    def __init__(self, params, device=0, handle=None):
        """handle: wrap a model that something else owns (a member of msqg_ensemble_create) instead of creating one"""
        self.L = lib()
        self.p = params
        self.N, self.nl = params.N, params.nl
        self.owned = handle is None
        if handle is None:
            h = C.c_void_p()
            check(self.L.msqg_create(C.byref(params), device, C.byref(h)))
        else:
            h = C.c_void_p(handle)
        self.h = h
        self.t = 0.0
        self.i = 0

    def close(self):
        if getattr(self, "h", None):
            if self.owned:
                self.L.msqg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def nfields(self, fid):
        return self.L.msqg_nfields(self.h, fid)

    def set(self, fid, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float64)
        assert arr.shape == (self.nfields(fid), self.N, self.N), (arr.shape, self.nfields(fid))
        check(self.L.msqg_set_field(self.h, fid, arr))

    def get(self, fid):
        out = np.zeros((self.nfields(fid), self.N, self.N))
        check(self.L.msqg_get_field(self.h, fid, out))
        return out

    def set_async(self, fid, pinned):
        """start the upload of a page-locked [nl][N][N] array (msqg_set_field_async); commit() hands it to the model"""
        check(self.L.msqg_set_field_async(self.h, fid, pinned))

    def commit(self):
        check(self.L.msqg_set_field_commit(self.h))

    def get_async(self, fid, pinned):
        """snapshot a list and start its download into a page-locked array (msqg_get_field_async)"""
        check(self.L.msqg_get_field_async(self.h, fid, pinned))

    def io_wait(self):
        check(self.L.msqg_io_wait(self.h))

    def set_smoother(self, name):
        """'lex': the reference's sweep order (default, parity path); 'rb': red-black ordering (throughput mode)"""
        check(self.L.msqg_set_smoother(self.h, {"lex": 0, "rb": 1}[name]))

    def set_energy_conserv(self, on):
        """the reference's -DENERGY_CONSERV=1 build (qg.h:310-373) as a runtime switch"""
        check(self.L.msqg_set_energy_conserv(self.h, int(bool(on))))

    def set_const(self):
        check(self.L.msqg_set_const(self.h))

    def invertq(self, q_id=Q):
        check(self.L.msqg_invertq(self.h, q_id))

    def comp_q(self):
        check(self.L.msqg_comp_q(self.h))

    def mgstats(self, mode=-1):
        s = MgStats()
        check(self.L.msqg_last_mgstats(self.h, mode, C.byref(s)))
        return s

    def test_cycles(self, nrelax, mode=-1):
        """len(nrelax) multigrid cycles, cycle k with nrelax[k] sweeps per level (msqg_test_cycles): the unknown (PSI, or
        plane `mode` of PM) is updated in place; returns the residual max norm after every cycle"""
        sched = np.ascontiguousarray(nrelax, dtype=np.int32)
        resa = np.zeros(len(sched))
        check(self.L.msqg_test_cycles(self.h, mode, sched, len(sched), resa))
        return resa

    def update(self, dtmax, q_id=Q):
        out = C.c_double()
        check(self.L.msqg_update(self.h, q_id, dtmax, C.byref(out)))
        return out.value

    def advance(self, out_id, in_id, dt):
        check(self.L.msqg_advance(self.h, out_id, in_id, dt))

    def step(self, tnext_event=-1.0):
        dt, tn = C.c_double(), C.c_double()
        check(self.L.msqg_step(self.h, self.t, tnext_event, C.byref(dt), C.byref(tn)))
        self.t = tn.value
        self.i += 1
        return dt.value

    def wavelet_filter(self, dtflt):
        """wavelet_filter(qol, pol, qofl, dtflt, nbar), msqg/qg.h:509-560"""
        check(self.L.msqg_wavelet_filter(self.h, dtflt))

    def filter_de(self, dtflt, ediag=None):
        check(self.L.msqg_filter_de(self.h, dtflt, float(self.p.ediag if ediag is None else ediag)))

    def energy_tend(self, dt, ediag=None):
        """energy_tend(pol, dt), msqg/qg_energy.h:228-242"""
        check(self.L.msqg_energy_tend(self.h, dt, float(self.p.ediag if ediag is None else ediag)))

    def reset_energy(self):
        check(self.L.msqg_reset_energy(self.h))

    def ke1(self):
        ke = C.c_double()
        check(self.L.msqg_ke1(self.h, C.byref(ke)))
        return ke.value

    def time_vcycle(self, nrelax=4, reps=5):
        ms = C.c_double()
        check(self.L.msqg_time_vcycle(self.h, nrelax, reps, C.byref(ms)))
        return ms.value

    PROF_CATS = ("relax_fine", "relax_coarse", "residual", "restrict", "prolong", "correct", "laplacian", "rhs", "exchange")

    def set_stream(self, cuda_stream):
        check(self.L.msqg_set_stream(self.h, C.c_void_p(cuda_stream)))

    def profile(self, on=True):
        check(self.L.msqg_profile_enable(self.h, 1 if on else 0))

    def profile_read(self):
        ms = (C.c_double * 9)(); cnt = (C.c_long * 9)(); aux = (C.c_long * 9)()
        check(self.L.msqg_profile_read(self.h, ms, cnt, aux))
        return {k: dict(ms=ms[i], count=cnt[i], aux=aux[i]) for i, k in enumerate(self.PROF_CATS)}

    @property
    def total_cycles(self):
        return self.L.msqg_total_cycles(self.h)

    @property
    def launches(self):
        return self.L.msqg_launch_count(self.h)
