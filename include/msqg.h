/*
 * msqg.h -- C ABI of the B200-native msqg multilayer-QG timestep.
 *
 * Two layers, both plain C (no C++/torch types cross this boundary):
 *
 *  (1) handle-based device layer `msqg_*`: what a host program binds to replace
 *      the reference's function-pointer plugin
 *          advance = advance_qg; update = update_qg;        (msqg/qg.h:922-923)
 *      and the solver/diagnostic calls around it.  All field buffers are HOST
 *      pointers to C-contiguous double [layer][y][x] (x fastest), the layout of
 *      pyset_field/pyget_field (msqg/qg.h:1164-1189); device memory is owned by
 *      the handle; calls are synchronous unless stated.
 *
 *  (2) the reference's own global-state surface (same names, same argument
 *      meaning as the SWIG module `qg`, msqg/qg.i:29-36, msqg/qg_bfn.i:10-46,
 *      and the driver msqg/qg.c): read_params, init_grid, set_vars, set_const,
 *      create_outdir, backup_config, trash_vars, set_vars_bfn, trash_vars_bfn,
 *      pystep_bfn, pyq2p, pyp2q, run.  Implemented in C on top of layer (1).
 *
 * Error behaviour: the reference calls exit(0) on fatal input errors
 * (msqg/qg.h:735-738,991-995,1009-1012); layer (1) returns a negative code
 * instead and layer (2) prints the reference's message and returns the code.
 * There is NO CPU fallback: every compute entry point fails with
 * MSQG_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef MSQG_H
#define MSQG_H

#ifdef __cplusplus
extern "C" {
#endif

#define MSQG_MAXL 32

enum {
  MSQG_OK = 0,
  MSQG_ERR_ARG = -1,     /* bad argument / unsupported configuration */
  MSQG_ERR_CUDA = -2,    /* CUDA failure or no device */
  MSQG_ERR_FILE = -3,    /* file missing (read_params, msqg/qg.h:735-738) */
  MSQG_ERR_CONFIG = -4,  /* thickness == 0 or Rom <= 0 (msqg/qg.h:990-1012) */
  MSQG_ERR_NOCONV = -5   /* informational: multigrid hit NITERMAX */
};

/* keys of params.in (msqg/qg.h:698-731) + derived values (:739-746) */
typedef struct msqg_params {
  int N, nl, ediag, varRo, nptr, flsrv;
  double L0, Rom, Ekb, Eks, tau0, Re, Re4, sbc, beta, afilt, Lfmax;
  double DT, tend, dtout, dtflt, CFL;
  double Fr[MSQG_MAXL], dh[MSQG_MAXL], upg[MSQG_MAXL], vpg[MSQG_MAXL];
  double iRe, iRe4;
  int stochastic;            /* the -D_STOCHASTIC build (msqg/qg.c:25) */
  double tr_stoch, itr_stoch, amp_stoch;
  int mode_pv_invert;        /* MODE_PV_INVERT (msqg/qg.h:4) as a runtime knob */
  /* passive tracers (nptr > 0), msqg/qg.h:98-106,726-727: relaxation time scale and Peclet number per tracer, and
     their inverses (:751-754) */
  double ptr_r[MSQG_MAXL], Pe[MSQG_MAXL], ptr_ir[MSQG_MAXL], iPe[MSQG_MAXL];
} msqg_params;

/* mgstats (Basilisk poisson.h; in-tree copy mspg/elliptic.h:118-123) */
typedef struct msqg_mgstats {
  int i;
  double resb, resa, sum;
  int nrelax;
} msqg_mgstats;

/* field-list ids for msqg_set_field / msqg_get_field */
enum {
  MSQG_PSI = 0,   /* pol      msqg/qg.h:24  */
  MSQG_Q,         /* qol      msqg/qg.h:23  */
  MSQG_PSIPG,     /* ppl      msqg/qg.h:36  */
  MSQG_FR,        /* Frl      msqg/qg.h:43  (nl scalars, nl-1 meaningful) */
  MSQG_QFORC,     /* q_forcl  msqg/qg.h:30  */
  MSQG_TOPO,      /* topo     msqg/qg.h:50  (1 scalar) */
  MSQG_RD,        /* Rd       msqg/qg.h:47  (1 scalar) */
  MSQG_SSTOCH,    /* s_stochl msqg/qg_stochastic.h:14 */
  MSQG_ZETA,      /* zetal    msqg/qg.h:25  */
  MSQG_DQ,        /* "updates" list of the predictor-corrector */
  MSQG_STR,       /* strl     msqg/qg.h:37  */
  MSQG_NSTOCH,    /* n_stochl msqg/qg_stochastic.h:13 */
  MSQG_IBU,       /* iBul     msqg/qg.h:42  */
  MSQG_CL2M,      /* cl2m     msqg/qg.h:40  (nl*nl scalars) */
  MSQG_CM2L,      /* cm2l     msqg/qg.h:41  */
  MSQG_PM,        /* pom      msqg/qg.h:33  */
  MSQG_QM,        /* qom      msqg/qg.h:32  */
  MSQG_TMP,       /* tmpl     msqg/qg.h:57  */
  MSQG_ZETAP,     /* zetapl   msqg/qg.h:26  */
  MSQG_QPRED,     /* "predictor" list of the predictor-corrector */
  MSQG_SIGFILT,   /* sig_filt msqg/qg.h:48  (1 scalar) */
  MSQG_DE_BF,     /* de_bfl   msqg/qg_energy.h:7   energy diagnostics (allocated on first use) */
  MSQG_DE_VD,     /* de_vdl   msqg/qg_energy.h:8  */
  MSQG_DE_J1,     /* de_j1l   msqg/qg_energy.h:9  */
  MSQG_DE_J2,     /* de_j2l   msqg/qg_energy.h:10 */
  MSQG_DE_J3,     /* de_j3l   msqg/qg_energy.h:11 */
  MSQG_DE_FT,     /* de_ftl   msqg/qg_energy.h:12 (accumulated by msqg_filter_de after every wavelet filter pass) */
  MSQG_PO_MFT,    /* po_mft   msqg/qg_energy.h:15 */
  MSQG_PTR,       /* ptracersl  msqg/qg.h:100 (nl*nptr scalars, index l*nptr + nt; zero-gradient boundaries) */
  MSQG_PTR_RELAX, /* ptr_relaxl msqg/qg.h:101 */
  MSQG_DPTR,      /* tracer part of `updates` */
  MSQG_QOF,       /* qofl     msqg/qg.h:27  filter mean (allocated on first use of the wavelet filter) */
  MSQG_SIGLEV,    /* sig_lev  msqg/qg.h:49  (finest level through get_field) */
  MSQG_NFIELDS
};

typedef struct msqg_model msqg_model;

/* ---- (1) handle-based device layer ------------------------------------ */

void msqg_default_params(msqg_params *p);
/* read_params (msqg/qg.h:689-761) into *p (which must hold defaults). */
int msqg_read_params(const char *path, msqg_params *p);

/* init_grid(N) + set_vars() (msqg/qg.h:837-925): allocates every layer list on
 * `device`, zero fields, ppl = vpg*x - upg*y, Frl = Fr.  N must be a power of
 * two >= 8, 2 <= nl <= 12.  sbc: 0 free slip, > 0 partial slip (qg.h:185-198), -1 doubly periodic (qg.h:842-846).
 * A periodic model is the tile of a 1 x 1 periodic group (layer 1b) that msqg_create builds by itself: N >= 16, the
 * red-black smoother, the layer-coupled inversion (stochastic forcing included) without tracers, energy diagnostics,
 * filter or a large-scale flow (the non-periodic psi_pg of qg.h:1105-1114); set_const / invertq / update / advance /
 * step / comp_q / set_field / get_field / ke1 behave as on a closed basin. */
int msqg_create(const msqg_params *p, int device, msqg_model **out);
void msqg_destroy(msqg_model *m);                 /* trash_vars, qg.h:1130-1154 */
/* run on this CUDA stream (a cudaStream_t passed as void*); default: own stream */
int msqg_set_stream(msqg_model *m, void *cuda_stream);
int msqg_nfields(msqg_model *m, int id);          /* scalars in list `id` (0 if absent) */
/* pyset_field (qg.h:1164-1175): host [nf][N][N] -> cells, then boundary() */
int msqg_set_field(msqg_model *m, int id, const double *host);
/* pyget_field (qg.h:1177-1189) */
int msqg_get_field(msqg_model *m, int id, double *host);
int msqg_set_flag_topo(msqg_model *m, int flag);  /* flag_topo, qg.h:971-977 */
/* Pipelined pyset_field / pyget_field for callers that advance a stream of independent states (ensemble members, the
 * forward / backward sweeps of msqg/qg_bfn.py): the PCIe transfers run on their own streams beside the step.
 *   msqg_set_field_async(m, id, in)  start the upload of in[nl][ny][nx]; returns at once (at most two in flight)
 *   msqg_set_field_commit(m)         the compute stream waits for the oldest upload and packs it into its list
 *   msqg_get_field_async(m, id, out) snapshot the list on the compute stream, start its download; returns at once
 *   msqg_io_wait(m)                  wait for every transfer started so far
 * id is MSQG_Q or MSQG_PSI.  Host buffers must be page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) and
 * must not be touched until msqg_io_wait (uploads: until their commit has been followed by a synchronising call).
 * Typical loop: set_field_async(in[0]); for k: { commit; set_field_async(in[k+1]); step; get_field_async(out[k]); } io_wait. */
int msqg_set_field_async(msqg_model *m, int id, const double *pinned_host);
int msqg_set_field_commit(msqg_model *m);
int msqg_get_field_async(msqg_model *m, int id, double *pinned_host);
int msqg_io_wait(msqg_model *m);
/* Ordering of the relaxation sweep inside mg_cycle.  0 (default): the reference's lexicographic in-place sweep
 * (relax_layer, msqg/poisson_layer.h:75-149, traversal of [BASILISK] foreach_level) -- results identical to a serial
 * reference build.  1: red-black ordering of the SAME cell update (cells with x+y even, then x+y odd), the
 * throughput mode: the reference itself documents that its sweep result depends on traversal order, OpenMP threads and
 * MPI decomposition (poisson_layer.h:55-65); red-black removes that dependence, so one result holds for 1..8 GPUs.
 * The iterate differs from the lexicographic one at the level of the solver tolerance (1e-3, qg.h:159).  Also set at
 * creation from the environment variable MSQG_SMOOTHER=rb. */
int msqg_set_smoother(msqg_model *m, int smoother);
int msqg_get_smoother(msqg_model *m);
/* The reference's compile-time variant -DENERGY_CONSERV=1 (msqg/qg.h:310-373, qg_energy.h:33-140) as a runtime switch:
 * advection_pv advects the full PV (jacobian(po, qot)) and drops J(psi_l, psi_l+1) from the stretching Jacobians,
 * advection_de books jacobian(po, comp_q(po)) in de_j1.  0 (default) is the default build of the reference.  Also set
 * at creation from the environment variable MSQG_ENERGY_CONSERV=1 (what `qcc -DENERGY_CONSERV=1` is to qg.e).  The
 * other compile-time switch of qg.h, _LS_RV = 0, needs no entry point: it is the arithmetic of flsrv = 0. */
int msqg_set_energy_conserv(msqg_model *m, int on);
int msqg_get_energy_conserv(msqg_model *m);
/* reset_layer_var (layer.h:37-41): zero the interior, ghost ring untouched */
int msqg_reset_field(msqg_model *m, int id);
/* layer thicknesses dhf (qg.h:895-896; overridden by dh_%dl.bin, qg.h:940-948) */
int msqg_set_dh(msqg_model *m, const double *dh);
int msqg_get_dh(msqg_model *m, double *dh);
/* set_const (qg.h:931-1116) minus the file reads (done by the C host, which
 * pushes file contents through msqg_set_field first) */
int msqg_set_const(msqg_model *m);

/* invertq(pol, q) (qg.h:113-163); q_id = MSQG_Q or MSQG_QPRED */
int msqg_invertq(msqg_model *m, int q_id);
int msqg_comp_q(msqg_model *m);                   /* comp_q(pol,qol), qg.h:396-403 */
/* mgstats of the last invertq; mode < 0: mgpsi (last solve), else modal solve */
int msqg_last_mgstats(msqg_model *m, int mode, msqg_mgstats *out);
long msqg_total_cycles(msqg_model *m);

/* update_qg(evolving=q_id, updates=DQ, dtmax) (qg.h:609-650); returns the new
 * dtmax through *dtmax_out (timestep() chain, qg.h:383-391). */
int msqg_update(msqg_model *m, int q_id, double dtmax, double *dtmax_out);
/* advance_qg(output, input, updates=DQ, dt) (qg.h:594-606) */
int msqg_advance(msqg_model *m, int out_id, int in_id, double dt);
/* one iteration of Basilisk run() (predictor-corrector.h), fused on device:
 *   dt = dtnext(update(q, DT)); qpred = q + dt/2*F(q); q += dt*F(qpred)
 * tnext < 0: no event rounding (dt = update's dtmax).  returns dt in *dt_out. */
int msqg_step(msqg_model *m, double t, double tnext, double *dt_out, double *tnext_out);
int msqg_ke1(msqg_model *m, double *ke);          /* writestdout, qg.c:101-106 */
/* multi-scale wavelet filter, msqg/qg.h:509-560: wavelet_filter(qol, pol, qofl, dtflt, nbar) as the `filter` event
 * calls it (:655-658).  q is replaced by its high-pass filtered version (scales below sig_filt = min(afilt*Rd, Lfmax)),
 * qofl receives (q_before - q_after)/dtflt.  nbar is passed by value in the reference, i.e. it is always 0. */
int msqg_wavelet_filter(msqg_model *m, double dtflt);
/* invertq(tmpl, qofl) of the output event (qg.c:124-129): the filtered-out stream function, left in MSQG_TMP */
int msqg_invert_filter_mean(msqg_model *m);
/* filter_de (qg_energy.h:207-226): second filter pass into tmp2l with -dtflt, de_ft += ..., po_mft = 0 */
int msqg_filter_de(msqg_model *m, double dtflt, double ediag);
/* the same with the running-mean slot named by the caller: pystep_de passes pol there (qg_energy.h:330), which zeroes
 * psi.  pm_field is MSQG_PO_MFT or MSQG_PSI. */
int msqg_filter_de_pm(msqg_model *m, double dtflt, double ediag, int pm_field);
/* energy diagnostics, msqg/qg_energy.h: energy_tend(pol, dt) of the comp_diag event (:228-242) with the weight
 * switch `ediag` (0: -psi*dq/dt, 1: dq/dt; qg.h:87).  The de_* lists are created on first use (set_vars_energy). */
int msqg_energy_tend(msqg_model *m, double dt, double ediag);
int msqg_reset_energy(msqg_model *m);             /* reset_layer_var(de_*), qg.c:158-164; also creates the lists */
/* the tendency of pystep_bfn (qg_bfn.h:21-80, vartype==1): q already set */
int msqg_tendency_bfn(msqg_model *m, double direction);
/* only the sign flips of pystep_bfn (qg_bfn.h:34-44) */
int msqg_bfn_direction(msqg_model *m, double direction);
/* timestep()'s static `previous` (Basilisk timestep.h): get / reset */
double msqg_get_ts_previous(msqg_model *m);
void msqg_set_ts_previous(msqg_model *m, double v);
/* seed of the host libc rand() stream used by the stochastic forcing
 * (qg_stochastic.h:9); noise is generated on the host in reference order */
void msqg_seed_noise(msqg_model *m, unsigned seed);
/* 0 (default): the noise field is drawn on the host from the libc rand() stream in the reference's traversal order
 * (bit-exact replay of qg_stochastic.h:117-126); 1: Philox4x32-10 on the device, same Box-Muller transform, order
 * independent -- the production mode of ensembles (seed from msqg_seed_noise) */
int msqg_set_noise_mode(msqg_model *m, int mode);
/* number of CUDA kernels launched by this handle since creation */
long msqg_launch_count(msqg_model *m);
const char *msqg_last_error(void);

/* keep the tendency list DQ when stepping with the fused msqg_step (default 0:
 * the RHS is consumed by the fused stage update and never stored) */
int msqg_set_keep_dq(msqg_model *m, int keep);
/* signed dissipation coefficients (pystep_bfn flips them, qg_bfn.h:34-44) */
int msqg_set_dissipation(msqg_model *m, double iRe, double iRe4, double Eks, double Ekb);
/* derived values of read_params (qg.h:739-746,757) for a hand-filled struct */
void msqg_derive_params(msqg_params *p);

/* kernel-level hooks for parity tests (level = multigrid level, n = 2^level):
 * fields are host [nf][n][n]; they exercise exactly the production kernels
 * with the model's stretching and layer metrics (set_const must have run). */
int msqg_test_relax(msqg_model *m, int level, double *a, const double *b, int nsweeps);
int msqg_test_relax_scalar(msqg_model *m, int level, double lambda, double *a, const double *b, int nsweeps);
int msqg_test_residual(msqg_model *m, const double *a, const double *b, double *res, double *maxres);
/* the residual pass of the multigrid solve with the restriction pyramid it leaves: mode < 0 the layer-coupled problem
 * (a, b [nl][n][n]), mode >= 0 the scalar Helmholtz problem of that vertical mode (mode_pv_invert, a, b [1][n][n]).
 * out receives res on levels D, D-1, .., *bottom one after another, each [nf][2^l][2^l] (at most 4/3 of level D) */
int msqg_test_residual_levels(msqg_model *m, int mode, const double *a, const double *b, double *out, double *maxres,
                              int *bottom);
int msqg_test_restrict(msqg_model *m, int level, const double *fine, double *coarse);
int msqg_test_prolong(msqg_model *m, int level, const double *coarse, double *fine);
/* div_by() (exact division by a pivot with known reciprocal) next to IEEE x/d */
int msqg_test_div(int device, const double *x, const double *d, double *q_fast, double *q_ieee, int n);
/* per-launch CUDA-event timing by kernel category (9 categories: relax finest,
 * relax coarser, residual, restrict, prolong, correct, laplacians, rhs, halo exchange) */
int msqg_profile_enable(msqg_model *m, int on);
int msqg_profile_read(msqg_model *m, double *ms, long *count, long *aux_sum);
/* per-worker timeline of one relax launch (debug): out[w] = {start ns, end ns, spins, 0} */
int msqg_test_relax_profile(msqg_model *m, int level, int nsweeps, long long *out, int max_workers);
/* one mg_cycle + residual at the model's shape, timed with CUDA events (ms) */
int msqg_time_vcycle(msqg_model *m, int nrelax, int reps, double *ms_out);

/* ---- (1c) ensembles of independent members on one device (BASELINE config 5; replicas only) ----
 * The reference runs one member per process (its own libc rand() stream, qg_stochastic.h:9,117-126).  Here the members
 * of a GPU are handles of one process, each with its own stream and noise stream; msqg_ensemble_step advances all of
 * them concurrently (one persistent host thread per member inside the library), member by member the bits of the
 * member run alone.  Fields go in and out through the member handles (msqg_set_field / msqg_get_field). */
typedef struct msqg_ensemble msqg_ensemble;
int msqg_ensemble_create(const msqg_params *p, int device, int nmembers, const unsigned *seeds /* NULL: 1000 + k */,
                         int noise_mode, int smoother, msqg_ensemble **out);
void msqg_ensemble_destroy(msqg_ensemble *e);
int msqg_ensemble_size(msqg_ensemble *e);
msqg_model *msqg_ensemble_member(msqg_ensemble *e, int k);
int msqg_ensemble_set_const(msqg_ensemble *e);                       /* set_const of every member */
int msqg_ensemble_step(msqg_ensemble *e, int nsteps, double *dt_last /* [nmembers] or NULL */);
double msqg_ensemble_time(msqg_ensemble *e, int k);

/* ---- (1b) 2-D domain decomposition: one tile per GPU, halo exchange == boundary() -------------
 * The semantics of the reference built with -D_MPI=1 (msqg/qg.c:12-19): px x py tiles on every
 * multigrid level whose global size is >= agg_n (coarser levels are agglomerated on tile (0,0)),
 * lexicographic Gauss-Seidel inside each tile with the neighbours' pre-sweep halo, halo exchange
 * after every sweep.  `local` keeps all tiles in one process on one device (tests / emulation),
 * `nccl` is one tile per process: rank = iy*px + ix, uid from msqg_nccl_unique_id on rank 0.
 * Field buffers are the TILE's [nf][ny][nx] block of the global [nf][N][N] array. */
typedef struct msqg_group msqg_group;
int msqg_nccl_unique_id(void *out128);
int msqg_group_create_local(const msqg_params *p, int device, int px, int py, int agg_n, msqg_group **out);
int msqg_group_create_nccl(const msqg_params *p, int device, int px, int py, int agg_n, int rank, int nranks,
                           const void *uid128, msqg_group **out);
/* Periodic boundaries (p->sbc == -1; red-black groups only): every side of every tile is an internal side and the
 * neighbour across a side of the domain is the tile on the opposite side (the tile itself where px or py is 1, in which
 * case msqg_group_create_local_sm accepts px = py = 1).  agg_n is chosen by the library from nl: every replicated level
 * is swept by the single-CTA coarse kernel with wrap-around neighbours, which holds levels up to 32^2 for nl <= 9 and
 * up to 16^2 for nl >= 10, so tiles start at 64^2 (nl <= 9) or 32^2 (nl >= 10) cells.  A red-black tile needs >= 16
 * cells per side there: at nl >= 10 a grid of 4 or more tiles across (4 x 2, 2 x 4, ...) is refused (MSQG_ERR_ARG).
 * The same with the smoother named (msqg_set_smoother): 1 = red-black.  A red-black group gives the bits of the
 * single-GPU red-black solve whatever px, py and agg_n are (a half-sweep is decomposition independent); levels with
 * fewer than agg_n cells per side are replicated on every GPU (all-gather of the restricted residual, redundant coarse
 * solve) and the sweeps of a distributed level need ONE halo exchange (deep halos, communication-avoiding).
 * Groups run the layer-coupled inversion; a closed-basin red-black group also runs the vertical-mode inversion
 * (p->mode_pv_invert) when the modes are uniform: varRo <= 0 and the same Fr on every tile (msqg_group_set_const checks
 * it).  Stochastic forcing (p->stochastic) runs on every group, periodic or closed, both smoothers: each tile draws its
 * window of the undecomposed noise field (Philox: global counter; libc: every tile replays the whole N^2 nl rand() stream,
 * O(N^2 nl) host time per draw and tile).  Seed every tile alike (msqg_seed_noise / msqg_set_noise_mode on each
 * msqg_group_tile, on every rank under NCCL): msqg_group_step refuses tiles that disagree on noise mode, seed or draw
 * count (MSQG_ERR_ARG).  Refused with MSQG_ERR_ARG: modal inversion on a lexicographic or periodic group. */
int msqg_group_create_local_sm(const msqg_params *p, int device, int px, int py, int agg_n, int smoother, msqg_group **out);
int msqg_group_create_nccl_sm(const msqg_params *p, int device, int px, int py, int agg_n, int smoother, int rank, int nranks,
                              const void *uid128, msqg_group **out);
int msqg_group_smoother(msqg_group *g);
/* 1: halos move by direct stores into the neighbours' memory (CUDA IPC over NVLink, dist_rb.cuh); 0: ncclSend/ncclRecv */
int msqg_group_transport(msqg_group *g);
void msqg_group_destroy(msqg_group *g);
int msqg_group_ntiles(msqg_group *g);                       /* tiles held by this process */
msqg_model *msqg_group_tile(msqg_group *g, int t);
int msqg_group_tile_info(msqg_group *g, int t, int *info6); /* ix, iy, x0, y0, nx, ny */
int msqg_group_set_field(msqg_group *g, int t, int id, const double *host_tile);
int msqg_group_get_field(msqg_group *g, int t, int id, double *host_tile);
int msqg_group_set_const(msqg_group *g);
int msqg_group_invertq(msqg_group *g, int q_id);
int msqg_group_step(msqg_group *g, double t, double tnext, double *dt_out, double *tnext_out);
int msqg_group_last_mgstats(msqg_group *g, msqg_mgstats *out);
/* as msqg_last_mgstats: mode < 0 the last solve, else the solve of that vertical mode (mode_pv_invert) */
int msqg_group_last_mode_mgstats(msqg_group *g, int mode, msqg_mgstats *out);
long msqg_group_total_cycles(msqg_group *g);
long msqg_group_exchanges(msqg_group *g);
long msqg_group_launches(msqg_group *g);
int msqg_group_set_stream_sync(msqg_group *g);
/* CUDA events on the group's stream: which 0 = start, 1 = stop + elapsed ms */
int msqg_group_timer(msqg_group *g, int which, double *ms);
int msqg_group_profile_enable(msqg_group *g, int on);
int msqg_group_profile_read(msqg_group *g, double *ms, long *count, long *aux_sum);

/* ---- (2) reference surface (global state, like the SWIG module `qg`) --- */

int read_params(char *path2file);                 /* qg.h:689 */
int init_grid(int n);                             /* Basilisk init_grid (qg.c:45) */
int set_vars(void);                               /* qg.h:837 */
int set_const(void);                              /* qg.h:931 (reads CWD input files) */
int create_outdir(void);                          /* qg.h:766 */
int backup_config(void);                          /* qg.h:782 */
int trash_vars(void);                             /* qg.h:1130 */
int set_vars_bfn(void);                           /* qg_bfn.h:7 */
int trash_vars_bfn(void);                         /* qg_bfn.h:12 */
int pystep_bfn(double *varin_py, int len1, int len2, int len3,
               double *tend_py, int len4, int len5, int len6,
               double direction, int vartype);    /* qg_bfn.h:21 */
int pyq2p(double *po_py, int len7, int len8, int len9,
          double *qo_py, int len10, int len11, int len12);   /* qg_bfn.h:85 */
int pyp2q(double *po_py, int len13, int len14, int len15,
          double *qo_py, int len16, int len17, int len18);   /* qg_bfn.h:95 */
int set_vars_energy(void);                        /* qg_energy.h:244 */
int trash_vars_energy(void);                      /* qg_energy.h:255 */
int pystep_de(double *po_py, int len1, int len2, int len3, double *de_bf_py, int len4, int len5, int len6,
              double *de_vd_py, int len7, int len8, int len9, double *de_j1_py, int len10, int len11, int len12,
              double *de_j2_py, int len13, int len14, int len15, double *de_j3_py, int len16, int len17, int len18,
              double *de_ft_py, int len19, int len20, int len21, int onlyKE);   /* qg_energy.h:294 (without filter_de) */
int run(void);                                    /* Basilisk run() + qg.c events */
/* access to the global handle/params behind the reference surface */
msqg_model *qg_model(void);
msqg_params *qg_params(void);
int qg_set_device(int device);
int qg_set_mode_pv_invert(int mode);              /* MODE_PV_INVERT, qg.h:4 */
int qg_set_stochastic(int on);                    /* -D_STOCHASTIC, qg.c:25 */
/* .bas files (auxiliar_input.h:24-59,101-149) on host arrays [nf][N][N] */
int qg_set_verbose(int v);
double qg_time(void);
int qg_iter(void);
const char *qg_outdir(void);
int qg_set_outdir(const char *d);
/* pieces of run(): init event (qg.c:53-72), event-loop reset, one iteration
 * (events + one step; returns 1 while running, 0 at the end, <0 on error) */
int qg_init_event(void);
int qg_run_reset(void);
int qg_run_iteration(int write_files);
int qg_write_bas(const char *name, int nf, int N, double L0, const double *v);
int qg_read_bas(const char *name, int nf, int N, double L0, double *v);

#ifdef __cplusplus
}
#endif
#endif
