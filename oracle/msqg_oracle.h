/*
 * msqg_oracle.h -- CPU oracle for the msqg multilayer QG timestep.
 *
 * TEST INFRASTRUCTURE ONLY.  This is a plain-C99 restatement of the reference
 * algorithm (bderembl/msom, msqg/qg.h + poisson_layer.h + eigmode.h + layer.h +
 * qg.c, and the Basilisk runtime pieces they call).  Only tests/, the
 * __graft_entry__.smoke() check and bench.py's cpu_baseline / --impl reference
 * legs may load it.  The product (msom_b200/) never links or calls it.
 *
 * PARITY UNPINNED: the reference ships no golden vectors or tests and cannot
 * be built here (qcc/Basilisk absent), so this oracle is pinned only by
 * known-answer identities (tests/test_oracle_*.py), not by reference outputs.
 *
 * Field API layout: C-contiguous double [layer][y][x] (x fastest), the layout
 * of pyset_field/pyget_field (msqg/qg.h:1164-1189).
 */
#ifndef MSQG_ORACLE_H
#define MSQG_ORACLE_H

#ifdef __cplusplus
extern "C" {
#endif

#define ORC_MAXL 32

typedef struct {
  /* keys of params.in, msqg/qg.h:698-731 */
  int N, nl, ediag, varRo, nptr, flsrv;
  double L0, Rom, Ekb, Eks, tau0, Re, Re4, sbc, beta, afilt, Lfmax;
  double DT, tend, dtout, dtflt, CFL;
  double Fr[ORC_MAXL], dh[ORC_MAXL], upg[ORC_MAXL], vpg[ORC_MAXL];
  /* derived, msqg/qg.h:739-746 */
  double iRe, iRe4;
  /* -D_STOCHASTIC build, msqg/qg_stochastic.h:3-6 */
  int stochastic;
  double tr_stoch, itr_stoch, amp_stoch;
  /* compile-time switch MODE_PV_INVERT (msqg/qg.h:4) made a runtime knob */
  int mode_pv_invert;
  /* passive tracers, msqg/qg.h:98-106,726-727,751-754: relaxation time scales and Peclet numbers per tracer */
  double ptr_r[ORC_MAXL], Pe[ORC_MAXL], ptr_ir[ORC_MAXL], iPe[ORC_MAXL];
  /* emulate Basilisk's MPI px*py block decomposition of the GS sweep
     (1,1 = serial reference order) */
  int px, py;
} orc_params;

typedef struct {
  int i;             /* cycles */
  double resb, resa; /* max residual before / after */
  double sum;        /* sum of rhs */
  int nrelax;        /* final nrelax */
} orc_mgstats;

typedef struct orc_model orc_model;

enum {
  ORC_PSI = 0, ORC_Q, ORC_PSIPG, ORC_FR, ORC_QFORC, ORC_TOPO, ORC_RD, ORC_SSTOCH,
  ORC_ZETA, ORC_DQ, ORC_STR, ORC_NSTOCH, ORC_IBU, ORC_CL2M, ORC_CM2L, ORC_PM, ORC_QM,
  ORC_TMP, ORC_ZETAP,
  /* energy diagnostics, msqg/qg_energy.h:7-15 */
  ORC_DE_BF, ORC_DE_VD, ORC_DE_J1, ORC_DE_J2, ORC_DE_J3, ORC_DE_FT, ORC_PO_MFT,
  /* passive tracers, msqg/qg.h:100-101: nl*nptr scalars, index l*nptr + nt */
  ORC_PTR, ORC_PTR_RELAX, ORC_DPTR,
  ORC_QOF, ORC_SIGLEV /* qofl (qg.h:27), sig_lev (qg.h:49; finest level through get_field) */
};

void orc_default_params(orc_params *p);
/* read_params, msqg/qg.h:689-761.  returns 0 ok, -1 file missing */
int orc_read_params(const char *path, orc_params *p);

orc_model *orc_create(const orc_params *p);      /* init_grid + set_vars */
void orc_destroy(orc_model *m);                  /* trash_vars */
int  orc_nfields(orc_model *m, int id);          /* number of scalars in list id */
void orc_set_field(orc_model *m, int id, const double *v); /* pyset_field */
void orc_get_field(orc_model *m, int id, double *v);       /* pyget_field */
int  orc_set_const(orc_model *m);                /* set_const; -1 on the exit(0) paths */
void orc_set_flag_topo(orc_model *m, int flag);
/* MPI-style block Gauss-Seidel emulation: px*py blocks on levels with n >= agg_n */
void orc_set_decomp(orc_model *m, int px, int py, int agg_n);
/* ordering of the relaxation sweep: 0 = the reference's lexicographic in-place sweep (default, the parity path);
   1 = red-black: the same cell update (poisson_layer.h:80-146) on the cells with (i+j) even, then on the cells with
   (i+j) odd.  The reference itself states that its sweep result depends on traversal order, OpenMP and MPI
   (poisson_layer.h:55-65); red-black removes that dependence (and ignores orc_set_decomp: it is decomposition
   independent).  It pins the throughput mode of the CUDA library (msqg_set_smoother). */
void orc_set_smoother(orc_model *m, int smoother);
/* stochastic forcing: 0 = the reference's sequential libc rand() draws (qg_stochastic.h:9,117-126; default),
   1 = counter-based Philox4x32-10 noise (production mode of the CUDA library: order independent, generated on the device) */
void orc_set_noise_mode(orc_model *m, int mode, unsigned seed);
void orc_test_philox(unsigned int *c4, unsigned int k0, unsigned int k1); /* Philox4x32-10 block function (known-answer tests) */
int orc_get_smoother(orc_model *m);
/* the reference's compile-time variant -DENERGY_CONSERV=1 as a runtime switch: advection_pv advects the full PV q
   instead of zeta + the stretching Jacobian J(psi_l, psi_l+1) (qg.h:310-312, :338-340, :366-367), and advection_de
   books J(psi, comp_q(psi)) in de_j1 (qg_energy.h:33-35, :64-66, :100-102, :132-134).  Not used by the stochastic
   advection_pv (qg_stochastic.h has no such branch).  _LS_RV = 0 needs no switch: it is flsrv = 0. */
void orc_set_energy_conserv(orc_model *m, int on);
void orc_init_noise(orc_model *m, unsigned seed);/* qg.c:60-70 with srand(seed) */
void orc_remove_mean_psi(orc_model *m);          /* qg.c:66-70 */

void orc_invertq(orc_model *m);                  /* invertq(pol,qol) */
void orc_comp_q(orc_model *m);                   /* comp_q(pol,qol) */
orc_mgstats orc_last_mgstats(orc_model *m, int mode);
int  orc_total_cycles(orc_model *m);
/* ncycles multigrid cycles with a fixed sweep schedule: cycle k relaxes nrelax[k] times per level, no tolerance stop and
   no nrelax adaptation; resa[k] is the residual max norm after cycle k.  mode = -1: the layer-coupled problem, PSI <- Q
   (the stretching restricted first, as invertq); mode = l (mode_pv_invert): plane l of PM <- QM (lambda restricted
   first).  The unknown is updated in place.  Returns -1 for a bad mode or an nrelax outside 2..100. */
int  orc_test_cycles(orc_model *m, int mode, const int *nrelax, int ncycles, double *resa);

/* update_qg on the model's q (evolving) -> DQ; returns dtmax */
double orc_update(orc_model *m, double dtmax);
/* one predictor-corrector step of Basilisk run() without the event machinery:
   dt = update(q, DT) (no dtnext rounding); returns dt used */
double orc_step(orc_model *m);
/* run() with events: output every dtout (invertq side effect), writestdout ke.
   write_files: 0 none, 1 write .bas into outdir.  returns number of steps. */
int orc_run(orc_model *m, int max_steps, int write_files, const char *outdir, int verbose);
double orc_time(orc_model *m);
double orc_ke1(orc_model *m);                    /* qg.c:101-106 */

/* wavelet_filter(qol, pol, qofl, dtflt, nbar), msqg/qg.h:509-560 (the `filter` event, :655-658) */
void orc_wavelet_filter(orc_model *m, double dtflt);
void orc_filter_de(orc_model *m, double dtflt);   /* filter_de, qg_energy.h:207-226, with the model's ediag */
/* sig_lev on level l (n = 2^l cells per side), [y][x] */
void orc_get_siglev(orc_model *m, int level, double *v);

/* energy diagnostics, msqg/qg_energy.h (ediag > -1): energy_tend(pol, dt) of the comp_diag event (:228-242,289-291);
   the lists are created on first use (set_vars_energy, :244-253).  filter_de needs the wavelet filter, which is
   out of scope: de_ft stays 0. */
void orc_energy_tend(orc_model *m, double dt);
void orc_reset_energy(orc_model *m);             /* reset_layer_var on the de_* lists, qg.c:158-164 */
/* pystep_de, qg_energy.h:294-340 (ediag = 1, dt = 1; without filter_de) */
void orc_pystep_de(orc_model *m, const double *po, double *de_bf, double *de_vd, double *de_j1, double *de_j2,
                   double *de_j3, double *de_ft, int onlyKE);

/* python entry points, msqg/qg_bfn.h */
void orc_pystep_bfn(orc_model *m, const double *q_in, double *tend, double direction, int vartype);
void orc_pyq2p(orc_model *m, double *po, const double *qo);
void orc_pyp2q(orc_model *m, const double *po, double *qo);

/* unit-level hooks for kernel parity tests (operate on scratch lists) */
/* one relax_layer sweep x nsweeps (each followed by boundary_level) on level l.
   a,b: [nl][n][n] arrays at that level; s: [nl-1][n][n] stretching at that level */
void orc_test_relax(int nl, int level, double L0, const double *dh, const double *s,
                    double *a, const double *b, int nsweeps, int px, int py);
double orc_test_residual(int nl, int level, double L0, const double *dh, const double *s,
                         const double *a, const double *b, double *res);
void orc_test_relax_rb(int nl, int level, double L0, const double *dh, const double *s,
                       double *a, const double *b, int nsweeps);
void orc_test_relax_scalar_rb(int level, double L0, const double *lam, double *a, const double *b, int nsweeps);
void orc_test_restrict(int nf, int level, const double *fine, double *coarse);
void orc_test_prolong(int nf, int level, const double *coarse, double *fine); /* level = fine level */
void orc_test_relax_scalar(int level, double L0, const double *lam, double *a, const double *b, int nsweeps);
double orc_test_residual_scalar(int level, double L0, const double *lam, const double *a, const double *b, double *res);
/* eigmod for one column: amat inputs -> cl2m[nl*nl], cm2l[nl*nl], iBu[nl]; returns 0 ok */
int orc_eigmod_column(int nl, const double *dhf, const double *Fr, double Ro,
                      double *cl2m, double *cm2l, double *iBu);

/* .bas I/O, msqg/auxiliar_input.h */
int orc_write_bas(const char *name, int nf, int N, double L0, const double *v /*[nf][y][x]*/);
int orc_read_bas(const char *name, int nf, int N, double L0, double *v);

#ifdef __cplusplus
}
#endif
#endif
