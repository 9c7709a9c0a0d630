/*
 * model.cu -- handle-based C ABI of the B200 msqg timestep (include/msqg.h, layer 1).
 *
 * Host logic here is the part of the reference that drives the hot kernels:
 *   mg_solve / mg_cycle      [BASILISK] poisson.h; in-tree copy mspg/elliptic.h:43-99,145-229
 *   poisson_layer            msqg/poisson_layer.h:263-306
 *   invertq                  msqg/qg.h:113-163
 *   update_qg / advance_qg   msqg/qg.h:594-650 (+ msqg/qg_stochastic.h)
 *   timestep()               [BASILISK] timestep.h; in-tree copy newqg/qg.h:202-219
 *   set_vars / set_const     msqg/qg.h:837-1116
 * No CPU fallback exists: every compute entry point needs a CUDA device.
 */
#include "../../include/msqg.h"
#include "layout.cuh"
#include "mg_kernels.cuh"
#include "rb_kernels.cuh"
#include "rhs_kernels.cuh"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <vector>
#include <utility>
#include <map>
#include <tuple>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <string>
#include <atomic>

static thread_local char g_err[512] = "";
static std::mutex g_kernel_init_mu; /* one-time per-device kernel setup (function attributes, occupancy queries) */
extern "C" const char *msqg_last_error(void) { return g_err; }
#define FAIL(code, ...)                        \
  do {                                         \
    snprintf(g_err, sizeof(g_err), __VA_ARGS__); \
    return (code);                             \
  } while (0)
#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) FAIL(MSQG_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
  } while (0)

static inline double sq(double x) { return x * x; }

enum { PROF_RELAX_FINE = 0, PROF_RELAX_COARSE, PROF_RESIDUAL, PROF_RESTRICT, PROF_PROLONG, PROF_CORRECT, PROF_LAP, PROF_RHS, PROF_XCHG, PROF_NCAT };

struct List {
  int nf = 0;
  double sg = -1.;               /* -1 dirichlet(0), +1 symmetry (layer.h:5-35) */
  double *lev[MSQG_MAXLEV + 1];  /* device pointers per level (only allocated levels non-NULL): row -1 of plane 0 */
  double *base[MSQG_MAXLEV + 1]; /* the allocations themselves (tiles carry extra frame rows below row -1, see msqg_model::fy);
                                    lev[] entries of two lists of the same level may be swapped, base[] entries stay */
  List() { for (auto &p : lev) p = nullptr; for (auto &p : base) p = nullptr; }
};

/* CUDA graphs of one multigrid cycle + residual (red-black smoother): the launch sequence of a cycle depends only on
 * nrelax, the problem (mode, unknown, right-hand side) and on which of the two da buffers is current on every level */
struct GraphEntry {
  cudaGraphExec_t exec = nullptr;
  std::vector<std::pair<int, int>> swaps; /* (tile, level) buffer swaps the cycle performs on the host side */
  long launches = 0, exchanges = 0;
};
typedef std::tuple<int, int, const void *, const void *, unsigned long long> GraphKey;
struct GraphCache {
  std::map<GraphKey, GraphEntry> entries;
  std::map<GraphKey, int> seen;
  void clear() { for (auto &e : entries) if (e.second.exec) cudaGraphExecDestroy(e.second.exec); entries.clear(); seen.clear(); }
};

struct msqg_model {
  msqg_params p;
  int N, nl, depth, device;
  /* tile of a px x py decomposition (single GPU: 1 x 1).  Levels < agg_level exist only on the tile that solves them
     for its process (tiles[0] of the group), as full square grids; finest tile is tnx x tny cells at (x0, y0). */
  int px, py, ix, iy, agg_level, tnx, tny, x0, y0;
  bool has_lev[MSQG_MAXLEV + 1];
  int fy[MSQG_MAXLEV + 1];     /* frame rows around the cells of a plane: 1 (the ghost ring) on undecomposed levels,
                                  MSQG_FRAME on the levels of a tile, which hold deep halos for the fused red-black sweeps
                                  (the row pitch then also keeps MSQG_FRAME columns on the right; MSQG_OX covers the left) */
  /* pipelined field I/O (msqg_set_field_async / msqg_get_field_async): two staging slots per direction, an upload and a
     download stream beside the compute stream, events for the hand-offs; created on first use */
  struct AsyncIO {
    cudaStream_t up = nullptr, down = nullptr;
    double *in_stage[2] = {nullptr, nullptr}, *out_stage[2] = {nullptr, nullptr};
    size_t cap = 0;                       /* doubles per staging slot */
    cudaEvent_t ev_up[2], ev_packed[2], ev_unpacked[2], ev_down[2];
    unsigned long up_count = 0, commit_count = 0, down_count = 0;
    int pending_id[2] = {-1, -1};
    bool ready = false;
  } io;
  struct msqg_group *group;    /* a periodic model made by msqg_create: the 1 x 1 group that owns this tile (else NULL) */
  int periodic;                /* sbc == -1 (periodic(right); periodic(top), qg.h:842-846): every side of every tile is an
                                  internal side whose halo comes from the opposite tile (or from the tile itself) */
  Geom gpatch;                 /* level agg_level-1 restricted to this tile (+ halo ring): scatter/gather scratch */
  double *da_patch, *res_patch; /* [nl] planes of gpatch */
  double *patch_stage;         /* contiguous gather / scatter block */
  size_t patch_doubles;
  double *xsend[9], *xrecv[9]; /* halo exchange: one buffer per neighbour direction (dist_rb.cuh), xcap doubles each */
  size_t xcap;
  /* peer-memory halo exchange (dist_rb.cuh): ONE allocation that neighbours map (CUDA IPC) and write into directly:
     [2 parities][9 directions][xcap] doubles of receive space, then 16 arrival flags, the exchange counter, block
     counters and an error word */
  double *xarea;
  size_t xarea_bytes;
  double *peer_area[9];        /* the neighbours' xarea (mapped), by direction; NULL where there is no neighbour */
  void *ipc_opened[9];
  double *gather_buf;          /* solver tile: gathered blocks of level agg_level-1, [px*py][nl][hy][hx] */
  cudaStream_t stream;
  bool own_stream;
  Geom g[MSQG_MAXLEV + 1];
  /* layer lists (finest level only unless noted) */
  List psi, q, qpred, dq, zeta, tmp, psipg, zetap, qforc, fr, str /*all levels*/, topo, rd, ro, sigfilt;
  List sstoch, nstoch;
  List qof, siglev, wvs, wvw, tmp2; /* wavelet filter: filter mean, sig_lev (all levels), restricted psi (levels < depth),
                                       coefficients (all levels), second filter mean of filter_de; on first use */
  int filter_vars;
  std::vector<double> h_sigfilt;   /* sig_filt on the finest level (host copy for sig_lev) */
  double siglev0;                  /* sig_lev of the root cell */
  List ptr, ptr_pred, dptr, ptr_relax; /* passive tracers, qg.h:100-101 (+ predictor and updates), nf = nl*nptr */
  List de_bf, de_vd, de_j1, de_j2, de_j3, de_ft, po_mft; /* energy diagnostics, qg_energy.h (allocated on first use) */
  int nme_ft, energy_vars;
  List da, res; /* all levels; nf = nl */
  List da2;     /* rb smoother: the relax pass is out of place (a CTA's output block is its neighbours' halo), da and da2 swap */
  List pm, qm, ibu /*all levels*/, cl2m, cm2l;
  double dhf[MSQG_MAXL], dhc[MSQG_MAXL], idh0[MSQG_MAXL], idh1[MSQG_MAXL];
  double iRe, iRe4, Eks, Ekb;
  int flag_topo, has_pg, has_zp, has_qforc;
  int const_set;
  /* uniform-stretching tables: s per level/layer and Thomas coefficients */
  double sbcc;                 /* partial slip coefficient of comp_del2 (qg.h:185-198), 0 = free slip */
  bool s_uniform;
  bool s_rowuniform;           /* stretching depends on y only (varRo > 0): per-row relax coefficients */
  double *rowcoef[MSQG_MAXLEV + 1]; /* device tables [rows][6][nl] or [rows][cols][6][nl] per level, or NULL */
  int coef_mx[MSQG_MAXLEV + 1], coef_my[MSQG_MAXLEV + 1]; /* margin of a table on the left / bottom side (tiles: the halo) */
  int coef_w[MSQG_MAXLEV + 1];  /* cells per row of a per-cell table (own cells + margins) */
  std::vector<double> s_lev;   /* [(depth+1)][nl] */
  std::vector<double> h_fr;    /* host copy of Frl finest [nl][N][N] */
  /* modal */
  bool modes_uniform;
  double h_cl2m[MSQG_NLMAX * MSQG_NLMAX], h_cm2l[MSQG_NLMAX * MSQG_NLMAX], h_ibu[MSQG_NLMAX];
  std::vector<double> lam_lev; /* [(depth+1)][nl] lambda per level (restricted) */
  /* horizontally varying Fr/Ro (eigmod per column, eigmode.h:74-299): lambda = iBu is a field, restricted to every
     level (poisson(): restriction({alpha, lambda}) [BASILISK]), and the scalar relax kernels read per-cell tables
     [ny][nx][6] = (0, 0, d, 1/d, 0, 0), d = -lambda*sq(Delta) + 2 + 2, one table per mode and level */
  double *modecoef[MSQG_NLMAX][MSQG_MAXLEV + 1];
  int coef_mode;               /* mode whose tables the scalar relax launches read; -1: constant lambda */
  /* scratch */
  double *d_stage;   /* staging [max nf][N][N] */
  size_t stage_doubles;
  double *d_scal;    /* device scalars: [0] maxres, [1..] umax[nl] */
  double *h_scal;    /* pinned mirror */
  double *d_wind;    /* [N] */
  double *d_kepart;
  unsigned long long *mailbox;
  size_t mailbox_words;
  int *d_err;
  int *h_err;
  long long *d_dbg; /* optional relax profiling buffer */
  int num_sms;
  /* state */
  double ts_previous;
  int corrector_step;
  /* libc rand() stream of this model (random_r on a TYPE_3 state == srand(seed); rand()) so that
     ensemble members in one process replay the sequence a one-member reference process would draw */
  struct random_data rng;
  char rng_state[128];
  std::vector<double> h_noise, h_sstoch;
  int noise_mode;               /* 0: host replay of the reference's libc rand() stream; 1: Philox on the device */
  unsigned int noise_seed;
  unsigned long long noise_draw; /* fields drawn since the last seed / mode change */
  int noise_agreed;             /* a group checked that its tiles agree on mode, seed and draw count (dist_impl.cuh) */
  double umax_pg[MSQG_MAXL];
  msqg_mgstats mgpsi, mgmode[MSQG_MAXL];
  long total_cycles, launches;
  int keep_dq;
  GraphCache graphs;
  std::vector<std::pair<int, int>> *swap_log; /* while a cycle is being recorded: (tile index, level) of every da/da2 swap */
  int tile_index;
  int use_graphs;
  int econs;       /* the reference's -DENERGY_CONSERV=1 build as a runtime switch (msqg_set_energy_conserv) */
  int smoother;    /* 0: reference-order (lexicographic) Gauss-Seidel, the parity path; 1: red-black ordering (rb_kernels.cuh) */
  int rb_reuse;    /* rb kernel: neighbours carried in registers (MSQG_RB_REUSE=0 switches it off, A/B tests) */
  /* optional per-launch timing (CUDA events on the model's stream) */
  int prof_on;
  std::vector<cudaEvent_t> prof_pool;
  struct ProfRec { int cat, aux; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof_recs;
  size_t prof_next;
};

struct ProfScope {
  msqg_model *m; cudaEvent_t e1; bool on;
  ProfScope(msqg_model *m_, int cat, int aux) : m(m_), e1(nullptr), on(m_->prof_on != 0) {
    if (!on) return;
    cudaEvent_t ev[2];
    for (int k = 0; k < 2; k++) {
      if (m->prof_next >= m->prof_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); m->prof_pool.push_back(e); }
      ev[k] = m->prof_pool[m->prof_next++];
    }
    cudaEventRecord(ev[0], m->stream);
    e1 = ev[1];
    m->prof_recs.push_back({cat, aux, ev[0], ev[1]});
  }
  ~ProfScope() { if (on) cudaEventRecord(e1, m->stream); }
};

/* ------------------------------------------------------------------ params */
extern "C" void msqg_default_params(msqg_params *p) {
  memset(p, 0, sizeof(*p));
  /* [BASILISK] N=64, L0=1, DT=1e10, CFL=0.5; msqg/qg.h:53-98 */
  p->N = 64; p->nl = 1; p->ediag = -1; p->L0 = 1.; p->beta = 0.5;
  p->afilt = 10.; p->Lfmax = 1.e10; p->DT = 1e10; p->tend = 1; p->dtout = 1;
  p->dtflt = -1; p->CFL = 0.5; p->amp_stoch = 1;
}

/* trim_whitespace, msqg/qg.h:668-675 (blanks only) */
static void trim_ws(char *s) {
  const char *d = s;
  do { while (*d == ' ') ++d; } while ((*s++ = *d++));
}
/* str2array, msqg/qg.h:678-687 */
static void str2array(char *s, double *arr) {
  int n = 0;
  char *p = strtok(s, "[,]");
  while (p != NULL && n < MSQG_MAXL) { arr[n++] = atof(p); p = strtok(NULL, ","); }
}
extern "C" void msqg_derive_params(msqg_params *p) {
  /* msqg/qg.h:739-746,757 */
  if (p->Re == 0) p->iRe = 0.; else p->iRe = 1 / p->Re;
  if (p->Re4 == 0) p->iRe4 = 0.; else p->iRe4 = -1 / p->Re4;
  if (p->Re != 0) p->DT = 0.5 * fmin(p->DT, sq(p->L0 / p->N) * p->Re / 4.);
  if (p->Re4 != 0) p->DT = 0.5 * fmin(p->DT, sq(sq(p->L0 / p->N)) * p->Re4 / 32.);
  if (p->tr_stoch != 0) p->itr_stoch = 1 / p->tr_stoch;
  for (int nt = 0; nt < p->nptr && nt < MSQG_MAXL; nt++) { /* qg.h:751-754 */
    if (p->ptr_r[nt] == 0) p->ptr_ir[nt] = 0.; else p->ptr_ir[nt] = 1 / p->ptr_r[nt];
    if (p->Pe[nt] == 0) p->iPe[nt] = 0.; else p->iPe[nt] = 1 / p->Pe[nt];
  }
}
extern "C" int msqg_read_params(const char *path, msqg_params *p) {
  FILE *fp = fopen(path, "rt");
  if (!fp) FAIL(MSQG_ERR_FILE, "file %s not found", path);
  char buf[300];
  while (fgets(buf, 300, fp)) {
    trim_ws(buf);
    char *k = strtok(buf, "=");
    char *v = strtok(NULL, "=");
    if (!k || !v) continue;
    if      (!strcmp(k, "N"))     p->N = atoi(v);
    else if (!strcmp(k, "nl"))    p->nl = atoi(v);
    else if (!strcmp(k, "ediag")) p->ediag = atoi(v);
    else if (!strcmp(k, "varRo")) p->varRo = atoi(v);
    else if (!strcmp(k, "nptr"))  p->nptr = atoi(v);
    else if (!strcmp(k, "flsrv")) p->flsrv = atoi(v);
    else if (!strcmp(k, "L0"))    p->L0 = atof(v);
    else if (!strcmp(k, "Rom"))   p->Rom = atof(v);
    else if (!strcmp(k, "Ekb"))   p->Ekb = atof(v);
    else if (!strcmp(k, "Eks"))   p->Eks = atof(v);
    else if (!strcmp(k, "tau0"))  p->tau0 = atof(v);
    else if (!strcmp(k, "Re"))    p->Re = atof(v);
    else if (!strcmp(k, "Re4"))   p->Re4 = atof(v);
    else if (!strcmp(k, "sbc"))   p->sbc = atof(v);
    else if (!strcmp(k, "beta"))  p->beta = atof(v);
    else if (!strcmp(k, "afilt")) p->afilt = atof(v);
    else if (!strcmp(k, "Lfmax")) p->Lfmax = atof(v);
    else if (!strcmp(k, "DT"))    p->DT = atof(v);
    else if (!strcmp(k, "tend"))  p->tend = atof(v);
    else if (!strcmp(k, "dtout")) p->dtout = atof(v);
    else if (!strcmp(k, "dtflt")) p->dtflt = atof(v);
    else if (!strcmp(k, "CFL"))   p->CFL = atof(v);
    else if (!strcmp(k, "Fr"))    str2array(v, p->Fr);
    else if (!strcmp(k, "dh"))    str2array(v, p->dh);
    else if (!strcmp(k, "upg"))   str2array(v, p->upg);
    else if (!strcmp(k, "ptr_r")) str2array(v, p->ptr_r);
    else if (!strcmp(k, "Pe"))    str2array(v, p->Pe);
    else if (!strcmp(k, "vpg"))   str2array(v, p->vpg);
    else if (p->stochastic && !strcmp(k, "tr_stoch"))  p->tr_stoch = atof(v);
    else if (p->stochastic && !strcmp(k, "amp_stoch")) p->amp_stoch = atof(v);
  }
  fclose(fp);
  msqg_derive_params(p);
  return MSQG_OK;
}

/* ------------------------------------------------------------------ allocation */
static int alloc_level(msqg_model *m, List &L, int nf, int l) {
  /* nf planes of (ny + 2 fy) rows; lev[] points at row -1 of plane 0; one frame of slack at the end so that
     "nf * plane doubles from lev[]" stays inside the allocation */
  const size_t off = (size_t)(m->fy[l] - 1) * m->g[l].pitch;
  const size_t bytes = ((size_t)nf * m->g[l].plane + 2 * off) * sizeof(double);
  CK(cudaMalloc(&L.base[l], bytes));
  CK(cudaMemsetAsync(L.base[l], 0, bytes, m->stream));
  L.lev[l] = L.base[l] + off;
  return MSQG_OK;
}
static int alloc_list(msqg_model *m, List &L, int nf, double sg, int lev_lo, int lev_hi) {
  L.nf = nf; L.sg = sg;
  for (int l = lev_lo; l <= lev_hi; l++) {
    if (!m->has_lev[l]) continue;
    int rc = alloc_level(m, L, nf, l);
    if (rc) return rc;
  }
  return MSQG_OK;
}
static void free_list(List &L) {
  for (auto &p : L.base) { if (p) cudaFree(p); p = nullptr; }
  for (auto &p : L.lev) p = nullptr;
  L.nf = 0;
}

static List *list_by_id(msqg_model *m, int id) {
  switch (id) {
    case MSQG_PSI: return &m->psi;     case MSQG_Q: return &m->q;
    case MSQG_PSIPG: return &m->psipg; case MSQG_FR: return &m->fr;
    case MSQG_QFORC: return &m->qforc; case MSQG_TOPO: return &m->topo;
    case MSQG_RD: return &m->rd;       case MSQG_SSTOCH: return &m->sstoch;
    case MSQG_ZETA: return &m->zeta;   case MSQG_DQ: return &m->dq;
    case MSQG_STR: return &m->str;     case MSQG_NSTOCH: return &m->nstoch;
    case MSQG_IBU: return &m->ibu;     case MSQG_CL2M: return &m->cl2m;
    case MSQG_CM2L: return &m->cm2l;   case MSQG_PM: return &m->pm;
    case MSQG_QM: return &m->qm;       case MSQG_TMP: return &m->tmp;
    case MSQG_ZETAP: return &m->zetap; case MSQG_QPRED: return &m->qpred;
    case MSQG_SIGFILT: return &m->sigfilt;
    case MSQG_DE_BF: return &m->de_bf; case MSQG_DE_VD: return &m->de_vd;
    case MSQG_DE_J1: return &m->de_j1; case MSQG_DE_J2: return &m->de_j2;
    case MSQG_DE_J3: return &m->de_j3; case MSQG_DE_FT: return &m->de_ft;
    case MSQG_PO_MFT: return &m->po_mft;
    case MSQG_QOF: return &m->qof; case MSQG_SIGLEV: return &m->siglev;
    case MSQG_PTR: return &m->ptr; case MSQG_PTR_RELAX: return &m->ptr_relax; case MSQG_DPTR: return &m->dptr;
  }
  return nullptr;
}

static dim3 grid2(int nx, int ny, dim3 b, int nz = 1) { return dim3((nx + b.x - 1) / b.x, (ny + b.y - 1) / b.y, nz); }
/* laplacian (+ face-speed reduction): two cells per thread when the tile width is even */
/* sbcc = sbc/((0.5*sbc+1)*sq(Delta)) for partial slip (qg.h:185-198), 0 for the free-slip default */
static void launch_lap(cudaStream_t st, int nf, const double *in, double *out, const Geom &g, double *umax, double sbcc) {
  if ((g.nx & 1) == 0) {
    dim3 b(32, 8);
    k_lap2<<<grid2(g.nx / 2, g.ny, b, nf), b, 0, st>>>(in, out, g, umax, sbcc);
  } else {
    dim3 b(64, 4);
    k_lap<<<grid2(g.nx + 1, g.ny + 1, b, nf), b, 0, st>>>(in, out, g, umax, sbcc);
  }
}
/* bilinear prolongation: one thread per coarse cell when the fine tile is exactly its 2 x 2 refinement */
static void launch_prolong(cudaStream_t st, int nf, const double *coarse, double *fine, const Geom &gc, const Geom &gf) {
  if (gf.nx == 2 * gc.nx && gf.ny == 2 * gc.ny) {
    dim3 b(32, 8);
    k_prolong4<<<grid2(gc.nx, gc.ny, b, nf), b, 0, st>>>(coarse, fine, gc, gf);
  } else {
    dim3 b(32, 8);
    k_prolong<<<grid2(gf.nx, gf.ny, b, nf), b, 0, st>>>(coarse, fine, gc, gf);
  }
}

static int pack_to(msqg_model *m, List &L, const double *host) {
  const Geom &g = m->g[m->depth];
  size_t cnt = (size_t)L.nf * g.nx * g.ny;
  if (cnt > m->stage_doubles) FAIL(MSQG_ERR_ARG, "staging buffer too small");
  CK(cudaMemcpyAsync(m->d_stage, host, cnt * sizeof(double), cudaMemcpyHostToDevice, m->stream));
  dim3 b(32, 8);
  k_pack<<<grid2(g.nx + 2, g.ny + 2, b, L.nf), b, 0, m->stream>>>(L.lev[m->depth], m->d_stage, L.nf, g, L.sg);
  m->launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(m->stream)); /* host buffer is borrowed for the call only */
  return MSQG_OK;
}
static int unpack_from(msqg_model *m, List &L, double *host) {
  const Geom &g = m->g[m->depth];
  size_t cnt = (size_t)L.nf * g.nx * g.ny;
  if (cnt > m->stage_doubles) FAIL(MSQG_ERR_ARG, "staging buffer too small");
  dim3 b(32, 8);
  k_unpack<<<grid2(g.nx, g.ny, b, L.nf), b, 0, m->stream>>>(m->d_stage, L.lev[m->depth], L.nf, g);
  m->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(host, m->d_stage, cnt * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  return MSQG_OK;
}

/* ------------------------------------------------------------------ create / destroy */
static void fill_geom_consts(Geom &g, double Delta) {
  g.Delta = Delta; /* == L0*(1./(1 << level)) [BASILISK], exact power-of-two scaling */
  g.rD = 1. / g.Delta;
  g.D2 = g.Delta * g.Delta; g.rD2 = 1. / g.D2;
  g.D12 = 12. * g.Delta * g.Delta; g.rD12 = 1. / g.D12;
  g.D2x = 2 * g.Delta; g.rD2x = 1. / g.D2x;
}

/* shared memory of the single-CTA coarse kernel k_coarse_rb, which keeps da and res of levels 1 .. Lc */
#define RB_COARSE_SMEM (200 * 1024)
/* the largest Lc (<= RB_COARSE_MAXLEV) whose levels 1 .. Lc fit into k_coarse_rb for nf planes: 5 (32^2) for nf <= 9,
 * 4 (16^2) for nf = 10 .. 12; 0 if not even levels 1 .. 2 fit */
static int coarse_max_level(int nf) {
  int Lc = RB_COARSE_MAXLEV;
  while (Lc >= 2) {
    size_t cells = 0;
    for (int l = 1; l <= Lc; l++) cells += (size_t)1 << (2 * l);
    if (2 * (size_t)nf * cells * sizeof(double) <= RB_COARSE_SMEM) break;
    Lc--;
  }
  return Lc >= 2 ? Lc : 0;
}

static int create_model(const msqg_params *p, int device, int px, int py, int ix, int iy, int agg_n, cudaStream_t shared,
                        msqg_model **out, int smoother = 0, bool coarse = true) {
  *out = nullptr;
  if (p->nl < 2 || p->nl > MSQG_NLMAX) FAIL(MSQG_ERR_ARG, "nl must be in [2,%d] (nl==1 is not functional in the reference)", MSQG_NLMAX);
  if (p->N < 8 || (p->N & (p->N - 1))) FAIL(MSQG_ERR_ARG, "N must be a power of two >= 8");
  const int per = p->sbc == -1;
  if (p->sbc < 0 && !per) FAIL(MSQG_ERR_ARG, "sbc is >= 0 (free / partial slip) or -1 (doubly periodic, qg.h:80)");
  if (per && smoother != 1)
    FAIL(MSQG_ERR_ARG, "periodic boundaries (sbc = -1) run on the tile machinery with the red-black smoother: "
                       "msqg_create does that by itself (a 1 x 1 group); tiles: msqg_group_create_local_sm(p, device, px, py, 0, 1, &group)");
  if (per && (p->mode_pv_invert || p->nptr > 0))
    FAIL(MSQG_ERR_ARG, "periodic boundaries are built for the layer-coupled path without tracers");
  for (int l = 0; per && l < p->nl; l++)
    if (p->upg[l] != 0 || p->vpg[l] != 0)
      FAIL(MSQG_ERR_ARG, "periodic boundaries with a large-scale flow (non-periodic psi_pg, qg.h:1105-1114) are not built");
  if (p->nptr < 0 || p->nptr > MSQG_MAXL) FAIL(MSQG_ERR_ARG, "nptr must be in 0..%d", MSQG_MAXL);
  if (p->nptr > 0 && p->stochastic) FAIL(MSQG_ERR_ARG, "passive tracers are not advanced by the stochastic advance_qg (qg_stochastic.h:139-147)");
  if (px < 1 || py < 1 || (px & (px - 1)) || (py & (py - 1))) FAIL(MSQG_ERR_ARG, "px, py must be powers of two");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    FAIL(MSQG_ERR_CUDA, "no CUDA device: the msqg timestep has no CPU path");
  if (device < 0 || device >= ndev) FAIL(MSQG_ERR_ARG, "bad device %d", device);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) FAIL(MSQG_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a", device, prop.major, prop.minor);
  msqg_model *m = new msqg_model();
  m->p = *p; m->N = p->N; m->nl = p->nl; m->device = device;
  m->num_sms = prop.multiProcessorCount;
  int depth = 0;
  while ((1 << depth) < p->N) depth++;
  m->depth = depth;
  { /* partial slip (sbc > 0), qg.h:185-198: coefficient of the vorticity ghosts, same expression as the reference */
    const double Delta = p->L0 / p->N;
    m->sbcc = p->sbc > 0 ? p->sbc / ((0.5 * p->sbc + 1) * sq(Delta)) : 0.;
  }
  m->px = px; m->py = py; m->ix = ix; m->iy = iy;
  m->agg_level = 0;
  m->periodic = per; m->group = nullptr;
  const bool tiled = px * py > 1 || per;
  if (per) {
    /* the replicated levels must all be swept by k_coarse_rb, the only kernel of those levels with wrap-around
       neighbours: levels up to 32^2 for nl <= 9, up to 16^2 for nl >= 10; everything above lives on tiles */
    const int top = 2 << coarse_max_level(p->nl);
    agg_n = p->N < top ? p->N : top;
  }
  if (px * py > 1 && p->sbc > 0) { msqg_destroy(m); FAIL(MSQG_ERR_ARG, "partial slip (sbc > 0) is not supported on decomposed grids"); }
  if (tiled) {
    int la = 1;
    while ((1 << la) < agg_n) la++;
    const char *why = nullptr;
    if (la > depth) why = "the agglomeration threshold exceeds N";
    else if (per && (((1 << la) / px) < MSQG_FRAME || ((1 << la) / py) < MSQG_FRAME)) {
      /* agg_n is not the caller's choice here: it is what the wrap-around coarse kernel holds for this nl */
      delete m;
      FAIL(MSQG_ERR_ARG, "a periodic %d^2 x nl=%d grid is replicated on every tile below its %d^2 level (what the wrap-around "
           "coarse kernel holds for this nl), so %d x %d tiles leave fewer than the %d cells per side a red-black tile needs there",
           p->N, p->nl, 1 << la, px, py, MSQG_FRAME);
    }
    else if (((1 << la) / px) < 8 || ((1 << la) / py) < 8) why = "tiles must keep >= 8 cells per side on every distributed level (raise agg_n)";
    else if (smoother == 1 && (((1 << la) / px) < MSQG_FRAME || ((1 << la) / py) < MSQG_FRAME))
      why = "red-black tiles must keep >= 16 cells per side on every distributed level (raise agg_n)";
    else if (la < 2) why = "agg_n too small";
    if (why) { delete m; FAIL(MSQG_ERR_ARG, "%s", why); }
    m->agg_level = la;
  }
  for (int l = 0; l <= depth; l++) {
    Geom &g = m->g[l];
    const bool dist = tiled && l >= m->agg_level;
    if (dist) {
      g.nx = (1 << l) / px; g.ny = (1 << l) / py;
      g.bc = (ix > 0 ? 1 : 0) | (ix < px - 1 ? 2 : 0) | (iy > 0 ? 4 : 0) | (iy < py - 1 ? 8 : 0);
      if (per) g.bc = 15;
      m->has_lev[l] = true;
      m->fy[l] = MSQG_FRAME;
      g.pitch = ((g.nx + MSQG_OX + MSQG_FRAME + 15) / 16) * 16;
    } else {
      g.nx = g.ny = 1 << l; g.bc = 0;
      m->has_lev[l] = coarse;
      m->fy[l] = 1;
      g.pitch = msqg_pitch(g.nx);
    }
    g.plane = (size_t)(g.ny + 2 * m->fy[l]) * g.pitch;
    fill_geom_consts(g, p->L0 / (1 << l));
  }
  m->tnx = m->g[depth].nx; m->tny = m->g[depth].ny;
  m->x0 = ix * m->tnx; m->y0 = iy * m->tny;
  m->da_patch = m->res_patch = m->patch_stage = nullptr;
  for (int k = 0; k < 9; k++) m->xsend[k] = m->xrecv[k] = nullptr;
  m->gather_buf = nullptr; m->xcap = 0; m->xarea = nullptr; m->xarea_bytes = 0;
  for (int k = 0; k < 9; k++) { m->peer_area[k] = nullptr; m->ipc_opened[k] = nullptr; }
  if (shared) { m->stream = shared; m->own_stream = false; }
  else {
    CK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    m->own_stream = true;
  }
  const int nl = p->nl, D = depth;
  int rc;
#define AL(L, nf, sg, lo, hi) if ((rc = alloc_list(m, L, nf, sg, lo, hi))) { msqg_destroy(m); return rc; }
  /* set_vars, msqg/qg.h:849-883: bc_type 0 -> dirichlet(0); +1 -> symmetry */
  AL(m->psi, nl, -1., D, D) AL(m->q, nl, -1., D, D) AL(m->qpred, nl, -1., D, D) AL(m->dq, nl, -1., D, D)
  if (p->nptr > 0) { /* qg.h:867-870: zero-gradient boundaries (bc_type + 1) */
    const int nt = nl * p->nptr;
    AL(m->ptr, nt, 1., D, D) AL(m->ptr_pred, nt, 1., D, D) AL(m->dptr, nt, 1., D, D) AL(m->ptr_relax, nt, 1., D, D)
  }
  AL(m->zeta, nl, -1., D, D) AL(m->tmp, nl, -1., D, D) AL(m->psipg, nl, -1., D, D) AL(m->zetap, nl, -1., D, D)
  AL(m->qforc, nl, -1., D, D) AL(m->fr, nl, 1., D, D) AL(m->str, nl, 1., 1, D)
  AL(m->topo, 1, 1., D, D) AL(m->rd, 1, 1., D, D) AL(m->ro, 1, 1., D, D) AL(m->sigfilt, 1, 1., D, D)
  AL(m->da, nl, -1., 1, D) AL(m->res, nl, -1., 1, D)
  if (p->mode_pv_invert) {
    AL(m->pm, nl, -1., D, D) AL(m->qm, nl, -1., D, D) AL(m->ibu, nl, 1., 1, D)
    AL(m->cl2m, nl * nl, 1., D, D) AL(m->cm2l, nl * nl, 1., D, D)
  }
  if (p->stochastic) { AL(m->sstoch, nl, -1., D, D) AL(m->nstoch, nl, -1., D, D) }
#undef AL
  int maxnf = p->mode_pv_invert ? nl * nl : nl;
  if (nl * p->nptr > maxnf) maxnf = nl * p->nptr;
  m->stage_doubles = (size_t)maxnf * m->tnx * m->tny;
  CK(cudaMalloc(&m->d_stage, m->stage_doubles * sizeof(double)));
  CK(cudaMalloc(&m->d_scal, 64 * sizeof(double)));
  CK(cudaHostAlloc(&m->h_scal, 64 * sizeof(double), cudaHostAllocMapped | cudaHostAllocPortable));
  CK(cudaMalloc(&m->d_wind, (size_t)p->N * sizeof(double)));
  CK(cudaMemsetAsync(m->d_wind, 0, (size_t)p->N * sizeof(double), m->stream));
  CK(cudaMalloc(&m->d_kepart, (size_t)((p->N + 15) / 16) * ((p->N + 15) / 16) * sizeof(double)));
  CK(cudaMalloc(&m->d_err, sizeof(int)));
  CK(cudaMemsetAsync(m->d_err, 0, sizeof(int), m->stream));
  CK(cudaHostAlloc(&m->h_err, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
  m->mailbox = nullptr; m->mailbox_words = 0; m->d_dbg = nullptr;
  m->nme_ft = 0; m->energy_vars = 0; m->filter_vars = 0; m->siglev0 = 0.;
  for (int l = 0; l <= MSQG_MAXLEV; l++) { m->rowcoef[l] = nullptr; m->coef_mx[l] = m->coef_my[l] = m->coef_w[l] = 0; }
  for (int k = 0; k < MSQG_NLMAX; k++) for (int l = 0; l <= MSQG_MAXLEV; l++) m->modecoef[k][l] = nullptr;
  m->coef_mode = -1; m->modes_uniform = true;
  m->s_rowuniform = false;
  for (int l = 0; l < nl; l++) m->dhf[l] = p->dh[l]; /* qg.h:895-896 */
  m->iRe = p->iRe; m->iRe4 = p->iRe4; m->Eks = p->Eks; m->Ekb = p->Ekb;
  m->ts_previous = 0.; m->corrector_step = 0;
  memset(&m->rng, 0, sizeof(m->rng));
  initstate_r(1u, m->rng_state, sizeof(m->rng_state), &m->rng); /* C default: srand(1) */
  m->flag_topo = 0; m->has_qforc = 0; m->has_zp = 0; m->const_set = 0;
  m->total_cycles = 0; m->launches = 0; m->keep_dq = 0; m->prof_on = 0; m->prof_next = 0;
  { const char *e = getenv("MSQG_SMOOTHER"); m->smoother = (e && !strcmp(e, "rb")) ? 1 : 0; }
  { const char *e = getenv("MSQG_ENERGY_CONSERV"); m->econs = (e && atoi(e) == 1) ? 1 : 0; }
  { const char *e = getenv("MSQG_RB_REUSE"); m->rb_reuse = (e && atoi(e) == 0) ? 0 : 1; }
  { const char *e = getenv("MSQG_GRAPH"); m->use_graphs = (e && atoi(e) == 0) ? 0 : 1; }
  m->swap_log = nullptr; m->tile_index = 0;
  m->noise_mode = 0; m->noise_seed = 1; m->noise_draw = 0; m->noise_agreed = 0;
  memset(&m->mgpsi, 0, sizeof(m->mgpsi));
  memset(m->mgmode, 0, sizeof(m->mgmode));
  memset(m->umax_pg, 0, sizeof(m->umax_pg));
  /* Frl = Frm, ppl = vpg*x - upg*y, Ro = Rom, Rd = 1, topo = 0 (qg.h:898-915) */
  {
    const int tx = m->tnx, ty = m->tny;
    const size_t tc = (size_t)tx * ty;
    const double Delta = p->L0 / p->N;
    std::vector<double> h((size_t)nl * tc, 0.);
    m->h_fr.assign((size_t)nl * tc, 0.);
    for (int l = 0; l < nl - 1; l++)
      for (size_t c = 0; c < tc; c++) m->h_fr[(size_t)l * tc + c] = p->Fr[l];
    if ((rc = pack_to(m, m->fr, m->h_fr.data()))) { msqg_destroy(m); return rc; }
    m->has_pg = 0;
    for (int l = 0; l < nl; l++) if (p->upg[l] != 0 || p->vpg[l] != 0) m->has_pg = 1;
    if (m->has_pg) {
      for (int l = 0; l < nl; l++)
        for (int j = 0; j < ty; j++)
          for (int i = 0; i < tx; i++) {
            const double x = (m->x0 + i + 0.5) * Delta, y = (m->y0 + j + 0.5) * Delta;
            h[((size_t)l * ty + j) * tx + i] = p->vpg[l] * x - p->upg[l] * y;
          }
      if ((rc = pack_to(m, m->psipg, h.data()))) { msqg_destroy(m); return rc; }
    }
    std::vector<double> one(tc, 1.);
    if ((rc = pack_to(m, m->rd, one.data()))) { msqg_destroy(m); return rc; }
  }
  if (tiled) { /* exchange / gather-scatter scratch */
    const int la = m->agg_level;
    Geom &gp = m->gpatch;
    gp.nx = m->g[la].nx / 2; gp.ny = m->g[la].ny / 2; gp.bc = 15;
    gp.pitch = msqg_pitch(gp.nx); gp.plane = (size_t)(gp.ny + 2) * gp.pitch;
    fill_geom_consts(gp, p->L0 / (1 << (la - 1)));
    CK(cudaMalloc(&m->da_patch, (size_t)nl * gp.plane * sizeof(double)));
    CK(cudaMalloc(&m->res_patch, (size_t)nl * gp.plane * sizeof(double)));
    CK(cudaMemsetAsync(m->da_patch, 0, (size_t)nl * gp.plane * sizeof(double), m->stream));
    CK(cudaMemsetAsync(m->res_patch, 0, (size_t)nl * gp.plane * sizeof(double), m->stream));
    m->patch_doubles = (size_t)nl * (gp.nx + 2) * (gp.ny + 2);
    CK(cudaMalloc(&m->patch_stage, m->patch_doubles * sizeof(double)));
    /* one exchange carries at most: MSQG_FRAME-wide halos of one list on every distributed level (sizes halve per level) */
    m->xcap = (size_t)nl * MSQG_FRAME * 2 * ((m->tnx > m->tny ? m->tnx : m->tny) + 2 * MSQG_FRAME);
    for (int k = 0; k < 9; k++) {
      if (k == 4) continue;
      CK(cudaMalloc(&m->xsend[k], m->xcap * sizeof(double)));
      CK(cudaMalloc(&m->xrecv[k], m->xcap * sizeof(double)));
    }
    if (coarse) CK(cudaMalloc(&m->gather_buf, (size_t)px * py * nl * gp.nx * gp.ny * sizeof(double)));
    m->xarea_bytes = (2 * 9 * m->xcap) * sizeof(double) + 4096;
    CK(cudaMalloc(&m->xarea, m->xarea_bytes));
    CK(cudaMemsetAsync(m->xarea, 0, m->xarea_bytes, m->stream));
  }
  CK(cudaStreamSynchronize(m->stream));
  *out = m;
  return MSQG_OK;
}

/* sbc = -1 through the single-model entry points: msqg_create builds a 1 x 1 periodic group (dist_impl.cuh) and hands out
   its tile; set_const / invertq / update / step / comp_q / destroy of that handle go through the group */
struct msqg_group;
static int pg_create(const msqg_params *p, int device, msqg_model **out);
static void pg_destroy(msqg_group *G);
static int pg_set_const(msqg_group *G);
static int pg_invertq(msqg_group *G, msqg_model *m, int q_id);
static int pg_update(msqg_group *G, msqg_model *m, int q_id, double dtmax, double *dtmax_out);
static int pg_step(msqg_group *G, msqg_model *m, double t, double tnext_event, double *dt_out, double *tnext_out);
static int pg_halo(msqg_group *G, int id);
static int pg_set_stream(msqg_group *G, cudaStream_t s);
static void io_teardown(msqg_model *m);

extern "C" int msqg_create(const msqg_params *p, int device, msqg_model **out) {
  if (p->sbc == -1) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) FAIL(MSQG_ERR_CUDA, "no CUDA device: the msqg timestep has no CPU path");
    return pg_create(p, device, out);
  }
  return create_model(p, device, 1, 1, 0, 0, 0, nullptr, out);
}

extern "C" void msqg_destroy(msqg_model *m) {
  if (!m) return;
  if (m->group) { msqg_group *G = m->group; m->group = nullptr; pg_destroy(G); return; } /* destroys this tile too */
  cudaSetDevice(m->device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  io_teardown(m);
  m->graphs.clear();
  List *all[] = {&m->psi, &m->q, &m->qpred, &m->dq, &m->zeta, &m->tmp, &m->psipg, &m->zetap, &m->qforc, &m->fr,
                 &m->str, &m->topo, &m->rd, &m->ro, &m->sigfilt, &m->sstoch, &m->nstoch, &m->da, &m->res,
                 &m->pm, &m->qm, &m->ibu, &m->cl2m, &m->cm2l, &m->da2,
                 &m->de_bf, &m->de_vd, &m->de_j1, &m->de_j2, &m->de_j3, &m->de_ft, &m->po_mft,
                 &m->ptr, &m->ptr_pred, &m->dptr, &m->ptr_relax, &m->qof, &m->siglev, &m->wvs, &m->wvw, &m->tmp2};
  for (List *L : all) free_list(*L);
  if (m->d_stage) cudaFree(m->d_stage);
  if (m->d_scal) cudaFree(m->d_scal);
  if (m->h_scal) cudaFreeHost(m->h_scal);
  if (m->d_wind) cudaFree(m->d_wind);
  if (m->d_kepart) cudaFree(m->d_kepart);
  if (m->d_err) cudaFree(m->d_err);
  if (m->h_err) cudaFreeHost(m->h_err);
  if (m->mailbox) cudaFree(m->mailbox);
  for (int l = 0; l <= MSQG_MAXLEV; l++) if (m->rowcoef[l]) cudaFree(m->rowcoef[l]);
  for (int k = 0; k < MSQG_NLMAX; k++) for (int l = 0; l <= MSQG_MAXLEV; l++) if (m->modecoef[k][l]) cudaFree(m->modecoef[k][l]);
  if (m->da_patch) cudaFree(m->da_patch);
  if (m->res_patch) cudaFree(m->res_patch);
  if (m->patch_stage) cudaFree(m->patch_stage);
  for (int k = 0; k < 9; k++) { if (m->xsend[k]) cudaFree(m->xsend[k]); if (m->xrecv[k]) cudaFree(m->xrecv[k]); }
  if (m->gather_buf) cudaFree(m->gather_buf);
  for (int k = 0; k < 9; k++) if (m->ipc_opened[k]) cudaIpcCloseMemHandle(m->ipc_opened[k]);
  if (m->xarea) cudaFree(m->xarea);
  for (cudaEvent_t e : m->prof_pool) cudaEventDestroy(e);
  if (m->own_stream && m->stream) cudaStreamDestroy(m->stream);
  delete m;
}

extern "C" int msqg_set_stream(msqg_model *m, void *s) {
  CK(cudaSetDevice(m->device));
  if (m->group) return pg_set_stream(m->group, (cudaStream_t)s); /* the group and its tile share one stream */
  CK(cudaStreamSynchronize(m->stream));
  m->graphs.clear();
  if (m->own_stream) cudaStreamDestroy(m->stream);
  m->stream = (cudaStream_t)s;
  m->own_stream = false;
  return MSQG_OK;
}
extern "C" int msqg_nfields(msqg_model *m, int id) {
  List *L = list_by_id(m, id);
  return (L && L->lev[m->depth]) ? L->nf : 0;
}
extern "C" long msqg_launch_count(msqg_model *m) { return m->launches; }
extern "C" long msqg_total_cycles(msqg_model *m) { return m->total_cycles; }
extern "C" double msqg_get_ts_previous(msqg_model *m) { return m->ts_previous; }
extern "C" void msqg_set_ts_previous(msqg_model *m, double v) { m->ts_previous = v; }
extern "C" int msqg_set_noise_mode(msqg_model *m, int mode) {
  if (mode != 0 && mode != 1) FAIL(MSQG_ERR_ARG, "noise mode is 0 (libc rand() replay) or 1 (Philox on the device)");
  m->noise_mode = mode; m->noise_draw = 0; m->noise_agreed = 0;
  return MSQG_OK;
}
extern "C" void msqg_seed_noise(msqg_model *m, unsigned seed) {
  m->noise_seed = seed; m->noise_draw = 0; m->noise_agreed = 0;
  memset(&m->rng, 0, sizeof(m->rng));
  initstate_r(seed, m->rng_state, sizeof(m->rng_state), &m->rng);
}
extern "C" int msqg_set_flag_topo(msqg_model *m, int flag) { m->flag_topo = flag; return MSQG_OK; }
extern "C" int msqg_set_smoother(msqg_model *m, int smoother) {
  if (smoother != 0 && smoother != 1) FAIL(MSQG_ERR_ARG, "smoother is 0 (reference order) or 1 (red-black)");
  if (m->periodic && smoother != 1) FAIL(MSQG_ERR_ARG, "periodic boundaries (sbc = -1) need the red-black smoother");
  m->smoother = smoother;
  m->graphs.clear();
  return MSQG_OK;
}
extern "C" int msqg_set_energy_conserv(msqg_model *m, int on) {
  if (on != 0 && on != 1) FAIL(MSQG_ERR_ARG, "energy_conserv is 0 or 1");
  m->econs = on;
  return MSQG_OK;
}
extern "C" int msqg_get_energy_conserv(msqg_model *m) { return m->econs; }
extern "C" int msqg_get_smoother(msqg_model *m) { return m->smoother; }
extern "C" int msqg_stretch_tables(msqg_model *m) {
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "the stretching path is decided by set_const");
  return m->s_uniform ? 0 : (m->s_rowuniform ? 1 : 2);
}
extern "C" int msqg_set_keep_dq(msqg_model *m, int keep) { m->keep_dq = keep; return MSQG_OK; }
extern "C" int msqg_set_dissipation(msqg_model *m, double iRe, double iRe4, double Eks, double Ekb) {
  m->iRe = iRe; m->iRe4 = iRe4; m->Eks = Eks; m->Ekb = Ekb; /* pystep_bfn flips these, qg_bfn.h:34-44 */
  return MSQG_OK;
}
extern "C" int msqg_set_dh(msqg_model *m, const double *dh) {
  for (int l = 0; l < m->nl; l++) m->dhf[l] = dh[l];
  return MSQG_OK;
}
extern "C" int msqg_get_dh(msqg_model *m, double *dh) {
  for (int l = 0; l < m->nl; l++) dh[l] = m->dhf[l];
  return MSQG_OK;
}
extern "C" int msqg_bfn_direction(msqg_model *m, double direction) {
  const double Re = m->p.Re, Re4 = m->p.Re4;
  if (direction > 0) {
    m->iRe = (Re == 0) ? 0. : 1 / Re; m->iRe4 = (Re4 == 0) ? 0. : -1 / Re4;
    m->Eks = fabs(m->Eks); m->Ekb = fabs(m->Ekb);
  } else {
    m->iRe = (Re == 0) ? 0. : -1 / Re; m->iRe4 = (Re4 == 0) ? 0. : 1 / Re4;
    m->Eks = -fabs(m->Eks); m->Ekb = -fabs(m->Ekb);
  }
  return MSQG_OK;
}
extern "C" int msqg_reset_field(msqg_model *m, int id) {
  CK(cudaSetDevice(m->device));
  List *L = list_by_id(m, id);
  if (!L || !L->lev[m->depth]) FAIL(MSQG_ERR_ARG, "field list %d is not allocated", id);
  const Geom &g = m->g[m->depth];
  for (int f = 0; f < L->nf; f++)
    CK(cudaMemset2DAsync(L->lev[m->depth] + (size_t)f * g.plane + GIDX(g.pitch, 0, 0), (size_t)g.pitch * sizeof(double), 0,
                         (size_t)g.nx * sizeof(double), g.ny, m->stream));
  return MSQG_OK;
}
extern "C" int msqg_last_mgstats(msqg_model *m, int mode, msqg_mgstats *out) {
  if (mode >= m->nl) FAIL(MSQG_ERR_ARG, "bad mode");
  *out = mode < 0 ? m->mgpsi : m->mgmode[mode];
  return MSQG_OK;
}

static int max_face_speed(msqg_model *m, List &L, double *umax_host);

extern "C" int msqg_set_field(msqg_model *m, int id, const double *host) {
  CK(cudaSetDevice(m->device));
  List *L = list_by_id(m, id);
  if (!L || !L->lev[m->depth]) FAIL(MSQG_ERR_ARG, "field list %d is not allocated", id);
  int rc = pack_to(m, *L, host);
  if (rc) return rc;
  const size_t cnt = (size_t)L->nf * m->tnx * m->tny;
  if (id == MSQG_FR) m->h_fr.assign(host, host + cnt);
  if (id == MSQG_SSTOCH) m->h_sstoch.assign(host, host + cnt);
  if (id == MSQG_PSIPG || id == MSQG_QFORC) {
    int nz = 0;
    for (size_t c = 0; c < cnt && !nz; c++) nz = host[c] != 0.;
    if (id == MSQG_PSIPG && nz && m->periodic)
      FAIL(MSQG_ERR_ARG, "periodic boundaries with a large-scale stream function (qg.h:1105-1114) are not built");
    if (id == MSQG_PSIPG) m->has_pg = nz; else m->has_qforc = nz;
  }
  return MSQG_OK;
}
extern "C" int msqg_get_field(msqg_model *m, int id, double *host) {
  CK(cudaSetDevice(m->device));
  List *L = list_by_id(m, id);
  if (!L || !L->lev[m->depth]) FAIL(MSQG_ERR_ARG, "field list %d is not allocated", id);
  return unpack_from(m, *L, host);
}

/* ------------------------------------------------------------------ pipelined field I/O
 * A caller that advances a stream of independent states (ensemble members, the forward / backward sweeps of
 * msqg/qg_bfn.py) can hide the PCIe time of pyset_field / pyget_field behind the step: the upload of the next state runs
 * on its own stream while the current one is stepped, the download of a result while the next one is stepped.  Host
 * buffers must be page-locked and stay untouched until msqg_io_wait (uploads: until the matching commit has run). */
static int io_setup(msqg_model *m) {
  msqg_model::AsyncIO &io = m->io;
  if (io.ready) return MSQG_OK;
  CK(cudaStreamCreateWithFlags(&io.up, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&io.down, cudaStreamNonBlocking));
  io.cap = (size_t)m->nl * m->tnx * m->tny;
  for (int k = 0; k < 2; k++) {
    CK(cudaMalloc(&io.in_stage[k], io.cap * sizeof(double)));
    CK(cudaMalloc(&io.out_stage[k], io.cap * sizeof(double)));
    CK(cudaEventCreateWithFlags(&io.ev_up[k], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&io.ev_packed[k], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&io.ev_unpacked[k], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&io.ev_down[k], cudaEventDisableTiming));
  }
  io.ready = true;
  return MSQG_OK;
}
static void io_teardown(msqg_model *m) {
  msqg_model::AsyncIO &io = m->io;
  if (!io.ready) return;
  cudaStreamSynchronize(io.up); cudaStreamSynchronize(io.down);
  for (int k = 0; k < 2; k++) {
    cudaFree(io.in_stage[k]); cudaFree(io.out_stage[k]);
    cudaEventDestroy(io.ev_up[k]); cudaEventDestroy(io.ev_packed[k]); cudaEventDestroy(io.ev_unpacked[k]); cudaEventDestroy(io.ev_down[k]);
  }
  cudaStreamDestroy(io.up); cudaStreamDestroy(io.down);
  io.ready = false;
}
static int io_list(msqg_model *m, int id, List **out) {
  if (id != MSQG_Q && id != MSQG_PSI) FAIL(MSQG_ERR_ARG, "asynchronous field I/O moves the evolving lists (MSQG_Q, MSQG_PSI)");
  List *L = list_by_id(m, id);
  if (!L || !L->lev[m->depth] || L->nf != m->nl) FAIL(MSQG_ERR_ARG, "field list %d is not allocated", id);
  *out = L;
  return MSQG_OK;
}
/* start the upload of host[nl][ny][nx] (pinned) for list `id`; returns at once.  At most two uploads may be in flight. */
extern "C" int msqg_set_field_async(msqg_model *m, int id, const double *pinned_host) {
  CK(cudaSetDevice(m->device));
  List *L;
  int rc;
  if ((rc = io_list(m, id, &L)) || (rc = io_setup(m))) return rc;
  msqg_model::AsyncIO &io = m->io;
  if (io.up_count - io.commit_count >= 2) FAIL(MSQG_ERR_ARG, "two uploads are already waiting for msqg_set_field_commit");
  const int slot = (int)(io.up_count & 1);
  if (io.up_count >= 2) CK(cudaStreamWaitEvent(io.up, io.ev_packed[slot], 0)); /* the slot's previous content has been packed */
  CK(cudaMemcpyAsync(io.in_stage[slot], pinned_host, io.cap * sizeof(double), cudaMemcpyHostToDevice, io.up));
  CK(cudaEventRecord(io.ev_up[slot], io.up));
  io.pending_id[slot] = id;
  io.up_count++;
  return MSQG_OK;
}
/* the compute stream waits for the oldest upload and packs it into its list (interior + ghost ring, as msqg_set_field) */
extern "C" int msqg_set_field_commit(msqg_model *m) {
  CK(cudaSetDevice(m->device));
  msqg_model::AsyncIO &io = m->io;
  if (!io.ready || io.commit_count >= io.up_count) FAIL(MSQG_ERR_ARG, "no upload to commit");
  const int slot = (int)(io.commit_count & 1);
  List *L;
  int rc;
  if ((rc = io_list(m, io.pending_id[slot], &L))) return rc;
  const Geom &g = m->g[m->depth];
  CK(cudaStreamWaitEvent(m->stream, io.ev_up[slot], 0));
  dim3 b(32, 8);
  k_pack<<<grid2(g.nx + 2, g.ny + 2, b, L->nf), b, 0, m->stream>>>(L->lev[m->depth], io.in_stage[slot], L->nf, g, L->sg);
  m->launches++;
  CK(cudaGetLastError());
  CK(cudaEventRecord(io.ev_packed[slot], m->stream));
  io.commit_count++;
  return MSQG_OK;
}
/* snapshot list `id` on the compute stream and start its download into host[nl][ny][nx] (pinned); returns at once */
extern "C" int msqg_get_field_async(msqg_model *m, int id, double *pinned_host) {
  CK(cudaSetDevice(m->device));
  List *L;
  int rc;
  if ((rc = io_list(m, id, &L)) || (rc = io_setup(m))) return rc;
  msqg_model::AsyncIO &io = m->io;
  const int slot = (int)(io.down_count & 1);
  const Geom &g = m->g[m->depth];
  if (io.down_count >= 2) CK(cudaStreamWaitEvent(m->stream, io.ev_down[slot], 0)); /* the slot's previous snapshot has left */
  dim3 b(32, 8);
  k_unpack<<<grid2(g.nx, g.ny, b, L->nf), b, 0, m->stream>>>(io.out_stage[slot], L->lev[m->depth], L->nf, g);
  m->launches++;
  CK(cudaGetLastError());
  CK(cudaEventRecord(io.ev_unpacked[slot], m->stream));
  CK(cudaStreamWaitEvent(io.down, io.ev_unpacked[slot], 0));
  CK(cudaMemcpyAsync(pinned_host, io.out_stage[slot], io.cap * sizeof(double), cudaMemcpyDeviceToHost, io.down));
  CK(cudaEventRecord(io.ev_down[slot], io.down));
  io.down_count++;
  return MSQG_OK;
}
/* wait for every transfer started so far (host buffers of downloads are valid afterwards) */
extern "C" int msqg_io_wait(msqg_model *m) {
  CK(cudaSetDevice(m->device));
  if (!m->io.ready) return MSQG_OK;
  CK(cudaStreamSynchronize(m->io.up));
  CK(cudaStreamSynchronize(m->io.down));
  return MSQG_OK;
}

/* ------------------------------------------------------------------ coefficients */
static LayerMetrics metrics_of(msqg_model *m) {
  LayerMetrics M;
  for (int l = 0; l < MSQG_NLMAX; l++) { M.idh0[l] = 0.; M.idh1[l] = 0.; }
  for (int l = 0; l < m->nl; l++) { M.idh0[l] = m->idh0[l]; M.idh1[l] = m->idh1[l]; }
  return M;
}

/* Thomas coefficients of relax_layer for horizontally uniform stretching
 * (poisson_layer.h:89-139, same expression order; host fp64 without FMA). */
template <int NL>
static RelaxCoef<NL> relax_coef_layers(msqg_model *m, int lev) {
  RelaxCoef<NL> C;
  const double Delta = m->g[lev].Delta;
  const double *s = &m->s_lev[(size_t)lev * m->nl];
  double t0[NL], t1[NL], t2[NL];
  for (int l = 0; l < NL; l++) { t0[l] = t1[l] = t2[l] = 0.; }
  if (NL > 1) {
    int ll = 0;
    t2[ll] = -sq(Delta) * s[ll] * m->idh1[ll];
    t1[ll] = -t2[ll];
    t1[ll] += 1. + 1.; t1[ll] += 1. + 1.;
    for (ll = 1; ll < NL - 1; ll++) {
      t0[ll] = -sq(Delta) * s[ll - 1] * m->idh0[ll];
      t2[ll] = -sq(Delta) * s[ll] * m->idh1[ll];
      t1[ll] = -t0[ll] - t2[ll];
      t1[ll] += 1. + 1.; t1[ll] += 1. + 1.;
    }
    ll = NL - 1;
    t0[ll] = -sq(Delta) * s[ll - 1] * m->idh0[ll];
    t1[ll] = -t0[ll];
    t1[ll] += 1. + 1.; t1[ll] += 1. + 1.;
    for (ll = 1; ll < NL; ll++) t1[ll] -= t0[ll] * t2[ll - 1] / t1[ll - 1];
  }
  for (int l = 0; l < NL; l++) { C.t0[l] = t0[l]; C.t2[l] = t2[l]; C.t1p[l] = t1[l]; C.rinv[l] = 1. / t1[l]; }
  for (int l = 0; l < NL; l++) { C.cf[l] = l > 0 ? t0[l] * C.rinv[l - 1] : 0.; C.cb[l] = t2[l] * C.rinv[l]; }
  C.msd2 = -sq(Delta);
  return C;
}
/* [BASILISK] poisson.h relax(): d = -lambda*sq(Delta) + 2 + 2 */
static RelaxCoef<1> relax_coef_scalar(msqg_model *m, int lev, double lambda) {
  RelaxCoef<1> C;
  const double Delta = m->g[lev].Delta;
  double d = -lambda * sq(Delta);
  d += 1. + 1.; d += 1. + 1.;
  C.t0[0] = 0.; C.t2[0] = 0.; C.t1p[0] = d; C.rinv[0] = 1. / d; C.cf[0] = C.cb[0] = 0.;
  C.msd2 = -sq(Delta);
  return C;
}

/* ------------------------------------------------------------------ relax launch */
/* coefficient table of the current relax launch: the stretching tables of the layer-coupled solver (k_rowcoef), or
   the lambda tables of one vertical mode (k_modecoef) while a scalar solve with a lambda FIELD is running */
static inline bool relax_table_per_cell(const msqg_model *m) { return m->coef_mode >= 0 || !m->s_rowuniform; }
/* ... as a pointer to the entry of own cell (0, 0): the stretching tables of a tile also cover its halo (margins) */
static inline const double *relax_table(const msqg_model *m, int lev) {
  if (m->coef_mode >= 0) return m->modecoef[m->coef_mode][lev];
  if (!m->rowcoef[lev]) return nullptr;
  const bool cell = relax_table_per_cell(m);
  return m->rowcoef[lev] + ((size_t)m->coef_my[lev] * (cell ? m->coef_w[lev] : 1) + (cell ? m->coef_mx[lev] : 0)) * 6 * m->nl;
}
/* entries per row of the table of relax_table (0: one entry per row) */
static inline int relax_table_stride(const msqg_model *m, int lev) {
  if (!relax_table_per_cell(m)) return 0;
  return m->coef_mode >= 0 ? m->g[lev].nx : m->coef_w[lev];
}
/* does a relax launch on NL coupled unknowns read tables (true) or per-level constants (false)? */
template <int NL>
static inline bool relax_uses_table(const msqg_model *m) { return NL > 1 ? !m->s_uniform : m->coef_mode >= 0; }
static int ensure_mailbox(msqg_model *m, size_t words) {
  if (words <= m->mailbox_words) return MSQG_OK;
  if (m->mailbox) { CK(cudaStreamSynchronize(m->stream)); CK(cudaFree(m->mailbox)); m->mailbox = nullptr; }
  CK(cudaMalloc(&m->mailbox, words * sizeof(unsigned long long)));
  /* arm every entry with the "empty" NaN payload: byte pattern is not uniform, use a fill kernel */
  m->mailbox_words = words;
  return MSQG_OK;
}
__global__ void k_fill_u64(unsigned long long *p, size_t n, unsigned long long v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

/* warp-specialised relax kernel (k_relax_ws): two warps per strip */
template <int NL, int K, int WPC, bool RCOEF = false>
static int launch_relax_ws_w(msqg_model *m, double *da, const double *res, int lev, int nsweeps, const RelaxCoef<NL> &C) {
  using Cfg = WsCfg<NL, K>;
  const Geom &g = m->g[lev];
  const int nworkers = (g.nx + K - 1 + Cfg::W - 1) / Cfg::W;
  const size_t words = (size_t)nworkers * K * g.ny * Cfg::NLP;
  if (words > m->mailbox_words) {
    const Geom &gf = m->g[m->depth];
    /* size it for the finest level with all nl layers: the launches on the coarser levels and modes reuse it */
    const size_t nlp = (size_t)((m->nl + 1) & ~1);
    size_t need = (size_t)((gf.nx + K - 1 + Cfg::W - 1) / Cfg::W) * K * gf.ny * nlp;
    if (words > need) need = words;
    int rc = ensure_mailbox(m, need);
    if (rc) return rc;
    k_fill_u64<<<m->num_sms * 4, 256, 0, m->stream>>>(m->mailbox, m->mailbox_words, MAIL_EMPTY);
    m->launches++;
    CK(cudaGetLastError());
  }
  RelaxArgs A;
  A.da = da; A.res = res; A.g = g; A.nsweeps = nsweeps;
  A.mailbox = m->mailbox; A.err = m->d_err; A.dbg = m->d_dbg; A.w_base = 0; A.rowcoef = RCOEF ? relax_table(m, lev) : nullptr;
  A.coef_cell = (RCOEF && relax_table_per_cell(m)) ? 1 : 0;
  if (RCOEF && (g.bc || !A.rowcoef)) FAIL(MSQG_ERR_ARG, "horizontally varying stretching (varRo, frpg) is supported on undecomposed levels only");
  const size_t smem = Cfg::smem_per_worker * WPC;
  const int tv = g.bc ? 1 : 0; /* variant: 0 plain, 1 tile (stored halos) */
  auto kern = RCOEF ? k_relax_ws<NL, K, WPC, false, RCOEF> : (tv ? k_relax_ws<NL, K, WPC, true> : k_relax_ws<NL, K, WPC, false>);
  /* per device (handles may live on several GPUs of one process): opt-in shared memory and co-resident CTAs per SM */
  static std::atomic<bool> attr_set_d[64][2];
  static int max_blocks_d[64][2] = {};
  std::atomic<bool> *attr_set = attr_set_d[m->device & 63];
  int *max_blocks = max_blocks_d[m->device & 63];
  std::unique_lock<std::mutex> init_lk(g_kernel_init_mu, std::defer_lock);
  if (!attr_set[tv].load(std::memory_order_acquire)) init_lk.lock(); /* first launches of several host threads: one sets up */
  if (!attr_set[tv].load(std::memory_order_relaxed)) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_blocks[tv], kern, 64 * WPC, smem));
    attr_set[tv].store(true, std::memory_order_release);
  }
  if (init_lk.owns_lock()) init_lk.unlock();
  const int grid = (nworkers + WPC - 1) / WPC;
  int cap = max_blocks[tv] * m->num_sms; /* co-resident CTAs (strips spin on their left neighbour) */
  { const char *e = getenv("MSQG_RELAX_CAP"); if (e && atoi(e) > 0 && atoi(e) < cap) cap = atoi(e); } /* tests: force panels */
  if (cap < 1) FAIL(MSQG_ERR_ARG, "relax kernel does not fit on the device (nl=%d)", NL);
  RelaxCoef<NL> Cc = C;
  /* a level wider than cap*WPC strips is swept in column panels, left to right: the last strip of a panel
     leaves its boundary column in the global mailbox, the first strip of the next launch picks it up */
  for (int b0 = 0; b0 < grid; b0 += cap) {
    A.w_base = b0 * WPC;
    const int nb = grid - b0 < cap ? grid - b0 : cap;
    void *args[] = {(void *)&A, (void *)&Cc};
    CK(cudaLaunchCooperativeKernel((void *)kern, dim3(nb), dim3(64 * WPC), args, smem, m->stream));
    m->launches++;
  }
  return MSQG_OK;
}
/* stretching that varies with y (varRo > 0): per-row coefficient tables, K = 4 instances only */
template <int NL>
static int launch_relax_rowcoef(msqg_model *m, double *da, const double *res, int lev, int nsweeps, const RelaxCoef<NL> &C) {
  if constexpr (NL <= 6) { /* instantiated for the layer counts the coupled solver is used with (build time) */
    constexpr size_t spw = WsCfg<NL, 4>::smem_per_worker;
    if constexpr (spw * 4 <= 220 * 1024) return launch_relax_ws_w<NL, 4, 4, true>(m, da, res, lev, nsweeps, C);
    else return launch_relax_ws_w<NL, 4, 2, true>(m, da, res, lev, nsweeps, C);
  } else {
    FAIL(MSQG_ERR_ARG, "varRo > 0 with the layer-coupled solver is built for nl <= 6 (nl = %d)", NL);
  }
}
template <int NL, int K>
static int launch_relax_ws(msqg_model *m, double *da, const double *res, int lev, int nsweeps, const RelaxCoef<NL> &C) {
  constexpr size_t spw = WsCfg<NL, K>::smem_per_worker;
  if constexpr (spw * 4 <= 220 * 1024) return launch_relax_ws_w<NL, K, 4>(m, da, res, lev, nsweeps, C);
  else if constexpr (spw * 2 <= 220 * 1024) return launch_relax_ws_w<NL, K, 2>(m, da, res, lev, nsweeps, C);
  else return launch_relax_ws_w<NL, K, 1>(m, da, res, lev, nsweeps, C);
}
template <int NL>
static int launch_relax_rb(msqg_model *m, double *da, const double *res, int lev, int nrelax, const RelaxCoef<NL> &C,
                           int halo, double *corr_a);
/* halo (red-black tiles): valid cells of deep halo on the internal sides, see launch_relax_rb */
template <int NL>
static int launch_relax(msqg_model *m, double *da, const double *res, int lev, int nrelax, const RelaxCoef<NL> &C,
                        int halo = 0, double *corr_a = nullptr) {
  if (m->smoother == 1) return launch_relax_rb<NL>(m, da, res, lev, nrelax, C, halo, corr_a);
  if (corr_a) FAIL(MSQG_ERR_ARG, "the correction is folded into red-black passes only");
  int done = 0;
  while (done < nrelax) {
    int ns = nrelax - done;
    int rc;
    /* k_relax_ws is instantiated for K = 4 only (build time): more than 4 sweeps are consecutive launches, which
       is the same arithmetic */
    if (ns > 4) ns = 4;
    if (relax_uses_table<NL>(m)) rc = launch_relax_rowcoef<NL>(m, da, res, lev, ns, C);
    else rc = launch_relax_ws<NL, 4>(m, da, res, lev, ns, C);
    if (rc) return rc;
    done += ns;
  }
  return MSQG_OK;
}


/* ------------------------------------------------------------------ red-black relax launch (rb_kernels.cuh) */
/* per-device launch state of one kernel instance: opt-in shared memory and co-resident CTAs per SM */
/* (handles of several host threads -- ensemble members -- may reach a kernel's first launch together: the one-time
   setup is double-checked under g_kernel_init_mu, the flag is published with release / read with acquire) */
struct KernelDevState { std::atomic<bool> set[64]; int occ[64][RB_NSMAX + 1]; }; /* only ever `static`: zero-initialised */
/* levels / tiles of at most lim^2 cells go through k_relax_rb_tile instead of the streaming k_relax_rb (nl <= 4) */
static bool rb_tiled(int nf, bool rcoef, long long cells) {
  if (nf > 4) return false;
  int lim = 512;
  { const char *e = getenv("MSQG_RB_TILE"); if (e) lim = atoi(e); }
  if (rcoef) { const char *e = getenv("MSQG_RB_COARSE_TABLES"); if (e && atoi(e) == 0) lim = 0; }
  return cells <= (long long)lim * lim;
}
template <int NL, bool RCOEF>
static int launch_relax_rb_pass(msqg_model *m, double *da, const double *res, int lev, int ns, const RelaxCoef<NL> &C,
                                const int *orange /* {ox_lo, ox_hi, oy_lo, oy_hi} */, int halo,
                                double *corr_a = nullptr /* k_relax_rb<..., FOLD = true>: a += da instead of da2 = da */) {
  using Cfg = RbCfg<NL>;
  const Geom &g = m->g[lev];
  const int nh = 2 * ns;
  if (da != m->da.lev[lev]) FAIL(MSQG_ERR_ARG, "the rb relax pass works on the model's da list");
  if (!m->da2.lev[lev]) { /* second buffer of the out-of-place pass, allocated on first use */
    int rc = alloc_level(m, m->da2, m->nl, lev);
    if (rc) return rc;
    m->da2.nf = m->nl;
  }
  RbArgs A;
  memset(&A, 0, sizeof(A));
  A.da = da; A.da_out = m->da2.lev[lev]; A.res = res; A.g = g; A.ns = ns;
  A.R = 2 * nh + 1 + RB_PF;
  A.TX = RB_WX - 2 * nh;
  A.ox_lo = orange[0]; A.ox_hi = orange[1]; A.oy_lo = orange[2]; A.oy_hi = orange[3];
  /* cells that exist: own cells, plus `halo` cells of deep halo on the sides that have a neighbouring tile */
  A.xlo = (g.bc & 1) ? -halo : 0; A.xhi = g.nx + ((g.bc & 2) ? halo : 0);
  A.ylo = (g.bc & 4) ? -halo : 0; A.yhi = g.ny + ((g.bc & 8) ? halo : 0);
  A.par0 = 0; /* tile origins are even on every distributed level (tiles keep >= 8 cells per side) */
  A.coef = RCOEF ? relax_table(m, lev) : nullptr;
  A.coef_cell = RCOEF ? relax_table_stride(m, lev) : 0;
  A.reuse = m->rb_reuse;
  if (RCOEF && !A.coef) FAIL(MSQG_ERR_ARG, "no coefficient table on level %d", lev);
  const int nxo_ = A.ox_hi - A.ox_lo, nyo_ = A.oy_hi - A.oy_lo;
  const bool fold = corr_a != nullptr;
  if (fold) {
    if (halo || g.bc || rb_tiled(NL, RCOEF, (long long)nxo_ * nyo_))
      FAIL(MSQG_ERR_ARG, "the correction is folded into streaming passes over a whole undecomposed level only");
    if (!rb_can_fold(NL)) FAIL(MSQG_ERR_ARG, "nl = %d has no folded relax pass", NL);
    A.a = corr_a;
  }
  if constexpr (NL <= 4) {
    /* small levels / tiles: one shared-memory window per CTA instead of the streaming pipeline (k_relax_rb_tile) */
    if (rb_tiled(NL, RCOEF, (long long)nxo_ * nyo_)) {
      constexpr int WS = RB_TO + 4 * RB_NSMAX;
      const size_t tsmem = (size_t)2 * NL * WS * WS * sizeof(double);
      auto tk = k_relax_rb_tile<NL, RCOEF>;
      static KernelDevState tst;
      const int dev = m->device & 63;
      if (!tst.set[dev].load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lk(g_kernel_init_mu);
        if (!tst.set[dev].load(std::memory_order_relaxed)) {
          CK(cudaFuncSetAttribute(tk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
          tst.set[dev].store(true, std::memory_order_release);
        }
      }
      RelaxCoef<NL> Cc = C;
      tk<<<dim3((nxo_ + RB_TO - 1) / RB_TO, (nyo_ + RB_TO - 1) / RB_TO), 512, tsmem, m->stream>>>(A, Cc);
      m->launches++;
      CK(cudaGetLastError());
      std::swap(m->da.lev[lev], m->da2.lev[lev]);
      if (m->swap_log) m->swap_log->push_back({m->tile_index, lev});
      return MSQG_OK;
    }
  }
  const size_t smem = (size_t)A.R * Cfg::row_bytes;
  const int threads = Cfg::NSMAX * RB_WX; /* fixed block: stages beyond nh only stream */
  auto kern = k_relax_rb<NL, RCOEF, false>;
  if constexpr (rb_can_fold(NL)) { if (fold) kern = k_relax_rb<NL, RCOEF, true>; }
  static KernelDevState sts[2];
  KernelDevState &st = sts[fold ? 1 : 0];
  const int dev = m->device & 63;
  if (!st.set[dev].load(std::memory_order_acquire)) {
    std::lock_guard<std::mutex> lk(g_kernel_init_mu);
    if (!st.set[dev].load(std::memory_order_relaxed)) {
      CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)((size_t)(4 * Cfg::NSMAX + 1 + RB_PF) * Cfg::row_bytes)));
      for (int s = 1; s <= Cfg::NSMAX; s++)
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&st.occ[dev][s], kern, Cfg::NSMAX * RB_WX,
                                                         (size_t)(4 * s + 1 + RB_PF) * Cfg::row_bytes));
      st.set[dev].store(true, std::memory_order_release);
    }
  }
  const int occ = st.occ[dev][ns] > 0 ? st.occ[dev][ns] : 1;
  const int nxo = A.ox_hi - A.ox_lo, nyo = A.oy_hi - A.oy_lo;
  const int nstrips = (nxo + A.TX - 1) / A.TX;
  /* row chunks: about one wave of CTAs; a chunk pays 2 nh halo rows + 2 nh pipeline steps, so keep it >= 32 rows */
  int nchunks = (m->num_sms * occ) / nstrips; /* never more CTAs than fit at once: a second, nearly empty wave doubles the time */
  if (nchunks > nyo / 32) nchunks = nyo / 32;
  if (nchunks < 1) nchunks = 1;
  A.rpc = (nyo + nchunks - 1) / nchunks;
  nchunks = (nyo + A.rpc - 1) / A.rpc;
  RelaxCoef<NL> Cc = C;
  kern<<<dim3(nstrips, nchunks), threads, smem, m->stream>>>(A, Cc);
  m->launches++;
  CK(cudaGetLastError());
  if (!fold) { /* a correcting pass writes no da: da and da2 stay as they were */
    std::swap(m->da.lev[lev], m->da2.lev[lev]);
    if (m->swap_log) m->swap_log->push_back({m->tile_index, lev});
  }
  return MSQG_OK;
}
/* nrelax sweeps as ceil(nrelax / NSMAX) passes of (almost) equal length; the result does not depend on the split.
 * halo (tiles, dist_rb.cuh): the deep halo holds `halo` valid cells on the internal sides on entry; each pass writes its
 * own cells plus what stays valid after its ns sweeps, halo - 2 ns cells, so the halo holds halo - 2 nrelax cells on
 * exit.  Without a halo on a level with internal sides only the own cells are swept.
 * corr_a (optional): the last pass adds da to this unknown instead of storing da (k_relax_rb<..., FOLD = true>). */
template <int NL>
static int launch_relax_rb(msqg_model *m, double *da, const double *res, int lev, int nrelax, const RelaxCoef<NL> &C,
                           int halo = 0, double *corr_a = nullptr) {
  constexpr int NSMAX = RbCfg<NL>::NSMAX;
  const Geom &g = m->g[lev];
  const bool deep = g.bc && halo > 0;
  int left = nrelax, h = halo;
  if (da != m->da.lev[lev]) FAIL(MSQG_ERR_ARG, "the rb relax pass works on the model's da list");
  while (left > 0) {
    const int passes = (left + NSMAX - 1) / NSMAX;
    const int ns = (left + passes - 1) / passes;
    const int ho = deep ? h - 2 * ns : 0;
    if (ho < 0) FAIL(MSQG_ERR_ARG, "halo of %d cells is too thin for %d sweeps", halo, nrelax);
    const int orange[4] = {(g.bc & 1) ? -ho : 0, g.nx + ((g.bc & 2) ? ho : 0), (g.bc & 4) ? -ho : 0, g.ny + ((g.bc & 8) ? ho : 0)};
    double *ca = left == ns ? corr_a : nullptr;
    int rc;
    if (relax_uses_table<NL>(m)) { /* horizontally varying stretching: tables over own cells + halo on tiles (g_stretching) */
      if constexpr (NL <= 6) rc = launch_relax_rb_pass<NL, true>(m, m->da.lev[lev], res, lev, ns, C, orange, h, ca);
      else FAIL(MSQG_ERR_ARG, "varRo > 0 with the layer-coupled solver is built for nl <= 6 (nl = %d)", NL);
    } else
      rc = launch_relax_rb_pass<NL, false>(m, m->da.lev[lev], res, lev, ns, C, orange, h, ca);
    if (rc) return rc;
    left -= ns; h = ho;
  }
  return MSQG_OK;
}

/* levels 1 .. Lc of a red-black cycle in one launch (k_coarse_rb): res[Lc] -> da[Lc].  Lc is chosen so that da and res
 * of all those levels fit in shared memory; 0 = not applicable (lexicographic smoother, varying stretching, tiny grids) */
static int coarse_top_level(msqg_model *m, int nf_problem, int maxlevel) {
  if (m->smoother != 1) return 0;
  /* horizontally varying stretching / lambda: the coarse kernel reads the coefficient tables (built for nl <= 6) */
  if (nf_problem > 1 && !m->s_uniform && (m->nl > 6 || !m->rowcoef[1] || m->g[1].bc)) return 0;
  if (nf_problem == 1 && !m->modes_uniform && !m->modecoef[0][1]) return 0;
  { const char *e = getenv("MSQG_RB_COARSE_TABLES"); /* A/B: tables through the level-by-level streaming kernel */
    if (e && atoi(e) == 0 && (nf_problem > 1 ? !m->s_uniform : !m->modes_uniform)) return 0; }
  if (!m->periodic) { const char *e = getenv("MSQG_RB_COARSE"); if (e && atoi(e) == 0) return 0; } /* A/B: level-by-level launches */
  int Lc = coarse_max_level(nf_problem);
  if (Lc > maxlevel) Lc = maxlevel;
  return Lc >= 2 ? Lc : 0;
}
template <int NL, bool RCOEF = false>
static int launch_coarse_rb(msqg_model *m, int Lc, int nrelax, const CoarseCoef<NL> &CC) {
  CoarseArgs A;
  memset(&A, 0, sizeof(A));
  A.res = m->res.lev[Lc]; A.da = m->da.lev[Lc]; A.g = m->g[Lc]; A.Lc = Lc; A.nrelax = nrelax; A.periodic = m->periodic;
  if (RCOEF) {
    for (int l = 1; l <= Lc; l++) {
      A.coef[l] = relax_table(m, l);
      if (!A.coef[l]) FAIL(MSQG_ERR_ARG, "no coefficient table on level %d", l);
    }
    A.coef_cell = relax_table_per_cell(m) ? 1 : 0;
  }
  size_t cells = 0;
  for (int l = 1; l <= Lc; l++) cells += (size_t)1 << (2 * l);
  const size_t smem = 2 * (size_t)NL * cells * sizeof(double);
  auto kern = k_coarse_rb<NL, RCOEF>;
  static KernelDevState st;
  const int dev = m->device & 63;
  if (!st.set[dev].load(std::memory_order_acquire)) {
    std::lock_guard<std::mutex> lk(g_kernel_init_mu);
    if (!st.set[dev].load(std::memory_order_relaxed)) {
      CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RB_COARSE_SMEM));
      st.set[dev].store(true, std::memory_order_release);
    }
  }
  CoarseCoef<NL> Cc = CC;
  kern<<<1, 512, smem, m->stream>>>(A, Cc);
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}

#define NL_CASE(n, ...) case n: { constexpr int NL = n; __VA_ARGS__; } break;
#define NL_SWITCH(nl, ...)                                  \
  switch (nl) {                                             \
    NL_CASE(2, __VA_ARGS__) NL_CASE(3, __VA_ARGS__) NL_CASE(4, __VA_ARGS__) NL_CASE(5, __VA_ARGS__)   \
    NL_CASE(6, __VA_ARGS__) NL_CASE(7, __VA_ARGS__) NL_CASE(8, __VA_ARGS__) NL_CASE(9, __VA_ARGS__)   \
    NL_CASE(10, __VA_ARGS__) NL_CASE(11, __VA_ARGS__) NL_CASE(12, __VA_ARGS__)                        \
    default: FAIL(MSQG_ERR_ARG, "unsupported nl=%d", nl);   \
  }

/* A few words from device memory to MAPPED pinned host memory, written by a kernel instead of a copy engine: the
 * convergence test of mg_solve, the CFL reduction and the error word are read back several times per step, and a
 * cudaMemcpyAsync of 8 bytes queues behind whatever bulk transfer occupies the device-to-host engine (the pipelined
 * field downloads of msqg_get_field_async: every read-back then waited ~10 ms for half a gigabyte to leave). */
template <class T>
__global__ void k_to_host(T *__restrict__ dst_mapped, const T *__restrict__ src, int n) {
  const int i = threadIdx.x;
  if (i < n) dst_mapped[i] = src[i];
  __threadfence_system();
}
template <class T>
static inline cudaError_t to_host(cudaStream_t st, T *host_mapped, const T *dev, int n) {
  k_to_host<T><<<1, 64, 0, st>>>(host_mapped, dev, n); /* n <= 64; pinned host memory is device-addressable (UVA) */
  return cudaGetLastError();
}

/* the few reduction words of a step are also CLEARED by a kernel: an asynchronous memset may be served by a copy engine
   and would then wait behind a bulk transfer exactly like the read-backs above */
__global__ void k_zero_words(double *p, int n) { if ((int)threadIdx.x < n) p[threadIdx.x] = 0.; }
static inline cudaError_t zero_words(cudaStream_t st, double *p, int n) {
  k_zero_words<<<1, 64, 0, st>>>(p, n);
  return cudaGetLastError();
}

static int check_relax_err(msqg_model *m) {
  CK(to_host(m->stream, m->h_err, m->d_err, 1));
  CK(cudaStreamSynchronize(m->stream));
  if (*m->h_err) {
    CK(cudaMemsetAsync(m->d_err, 0, sizeof(int), m->stream));
    k_fill_u64<<<m->num_sms * 4, 256, 0, m->stream>>>(m->mailbox, m->mailbox_words, MAIL_EMPTY);
    FAIL(MSQG_ERR_CUDA, "relax wavefront timed out waiting on a neighbour strip");
  }
  return MSQG_OK;
}

/* ------------------------------------------------------------------ multigrid */
struct MgProblem {
  int nf;            /* nl (layer-coupled) or 1 (one vertical mode) */
  int mode;          /* -1 layer-coupled, else mode index */
  double *a;         /* finest-level unknown, nf planes, ghosts maintained */
  const double *b;   /* finest-level rhs */
};

/* Lowest level of res that mg_residual_enqueue leaves restricted: on one undecomposed, non-periodic grid the residual
 * kernel also writes the restriction pyramid of its 32x32 tiles, levels D-1 .. D-5, never below level 1 (minlevel = 1:
 * level 0 is not read).  Elsewhere it writes level D only. */
static int residual_pyr_bottom(const msqg_model *m) {
  const int D = m->depth;
  if (m->g[D].bc != 0 || m->periodic || D < 2) return D;
  return D - PYR_MAXLEV > 1 ? D - PYR_MAXLEV : 1;
}

/* res = b - A a on level D and its max norm in d_scal[0], without the restriction pyramid (one grid or one tile) */
static int launch_residual(msqg_model *m, const MgProblem &P) {
  const int D = m->depth;
  const Geom &g = m->g[D];
  CK(zero_words(m->stream, m->d_scal, 1));
  dim3 b(64, 4);
  { ProfScope ps(m, PROF_RESIDUAL, 0);
  if (P.mode < 0) {
    LayerMetrics M = metrics_of(m);
    NL_SWITCH(m->nl, k_residual<NL><<<grid2(g.nx, g.ny, b), b, 0, m->stream>>>(P.a, P.b, m->res.lev[D], m->str.lev[D], g, M, m->d_scal));
  } else {
    k_residual_scalar<<<grid2(g.nx, g.ny, b), b, 0, m->stream>>>(P.a, P.b, m->res.lev[D], m->ibu.lev[D] + (size_t)P.mode * g.plane, g, m->d_scal);
  }
  }
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}
static int mg_residual_enqueue(msqg_model *m, const MgProblem &P) {
  const int D = m->depth;
  const Geom &g = m->g[D];
  const int bottom = residual_pyr_bottom(m);
  if (bottom < D) {
    CK(zero_words(m->stream, m->d_scal, 1));
    PyrLevels L;
    L.nlev = D - bottom;
    for (int k = 0; k < PYR_MAXLEV; k++) {
      const int l = k < L.nlev ? D - 1 - k : D;
      L.p[k] = m->res.lev[l]; L.pitch[k] = m->g[l].pitch; L.plane[k] = m->g[l].plane; L.n[k] = m->g[l].nx;
    }
    const dim3 b(32, 8), grid((g.nx + PYR_TILE - 1) / PYR_TILE, (g.ny + PYR_TILE - 1) / PYR_TILE);
    const LayerMetrics M = metrics_of(m);
    StretchConsts S;
    for (int l = 0; l < MSQG_NLMAX; l++) S.s[l] = l < m->nl ? m->s_lev[(size_t)D * m->nl + l] : 0.;
    { ProfScope ps(m, PROF_RESIDUAL, 0);
    if (P.mode >= 0) {
      k_residual_pyr<1, true><<<grid, b, 0, m->stream>>>(P.a, P.b, m->res.lev[D], m->ibu.lev[D] + (size_t)P.mode * g.plane, S, g, M, L, m->d_scal);
    } else if (m->s_uniform) { /* s_lev holds the field's one value per layer, bit for bit */
      NL_SWITCH(m->nl, k_residual_pyr<NL, false><<<grid, b, 0, m->stream>>>(P.a, P.b, m->res.lev[D], nullptr, S, g, M, L, m->d_scal));
    } else {
      NL_SWITCH(m->nl, k_residual_pyr<NL, true><<<grid, b, 0, m->stream>>>(P.a, P.b, m->res.lev[D], m->str.lev[D], S, g, M, L, m->d_scal));
    }
    }
    m->launches++;
    CK(cudaGetLastError());
  } else {
    int rc = launch_residual(m, P);
    if (rc) return rc;
  }
  CK(to_host(m->stream, m->h_scal, m->d_scal, 1));
  return MSQG_OK;
}
/* the residual norm that mg_residual_enqueue left in the pinned mirror */
static int mg_residual_read(msqg_model *m, double *maxres) {
  CK(cudaStreamSynchronize(m->stream));
  *maxres = m->h_scal[0];
  return MSQG_OK;
}
static int mg_residual(msqg_model *m, const MgProblem &P, double *maxres) {
  int rc = mg_residual_enqueue(m, P);
  if (rc) return rc;
  return mg_residual_read(m, maxres);
}

/* Run `body` (which only enqueues work on `st`) through a CUDA graph: the first use of a key runs eagerly (lazy
 * allocations, function attributes), the second records and instantiates, later uses replay.  The host-side effects of
 * the body -- da/da2 buffer swaps, launch counters -- are logged while recording and re-applied on replay. */
template <class F>
static int run_graphed(cudaStream_t st, GraphCache &gc, const GraphKey &key, std::vector<msqg_model *> &models, long *exchanges, bool enabled,
                       F body) {
  if (!enabled) return body();
  auto it = gc.entries.find(key);
  if (it != gc.entries.end()) {
    GraphEntry &E = it->second;
    CK(cudaGraphLaunch(E.exec, st));
    for (auto &sw : E.swaps) { msqg_model *m = models[sw.first]; std::swap(m->da.lev[sw.second], m->da2.lev[sw.second]); }
    models[0]->launches += E.launches;
    if (exchanges) *exchanges += E.exchanges;
    return MSQG_OK;
  }
  if (gc.seen[key]++ == 0) return body();
  GraphEntry E;
  long l0 = 0, x0 = exchanges ? *exchanges : 0;
  for (msqg_model *m : models) { l0 += m->launches; m->swap_log = &E.swaps; }
  cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed);
  int rc = e == cudaSuccess ? body() : MSQG_ERR_CUDA;
  cudaGraph_t g = nullptr;
  cudaError_t e2 = cudaStreamEndCapture(st, &g);
  long l1 = 0;
  for (msqg_model *m : models) { l1 += m->launches; m->swap_log = nullptr; }
  if (e != cudaSuccess || rc || e2 != cudaSuccess || !g) {
    if (g) cudaGraphDestroy(g);
    cudaGetLastError();
    if (rc) return rc;
    FAIL(MSQG_ERR_CUDA, "recording the multigrid cycle as a CUDA graph failed: %s", cudaGetErrorString(e != cudaSuccess ? e : e2));
  }
  e = cudaGraphInstantiate(&E.exec, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) FAIL(MSQG_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e));
  E.launches = l1 - l0; E.exchanges = exchanges ? *exchanges - x0 : 0;
  CK(cudaGraphLaunch(E.exec, st));
  gc.entries[key] = E;
  return MSQG_OK;
}
static unsigned long long da_parity_mask(msqg_model *m) {
  unsigned long long mask = 0;
  for (int l = 1; l <= m->depth; l++)
    if (m->da.lev[l] && m->da.base[l] && m->da.lev[l] != m->da.base[l] + (size_t)(m->fy[l] - 1) * m->g[l].pitch) mask |= 1ull << l;
  return mask;
}

/* restriction of res from level `from` down to level 1, then the up-leg of the cycle on levels 1 .. top (da = 0 on
 * level 1, bilinear prolongation, nrelax sweeps).  With the red-black smoother the levels up to 32^2 run as ONE launch
 * (k_coarse_rb), which also does their restrictions. */
/* MSQG_RB_FOLD=0: a separate k_correct launch instead of the correction folded into the last relax pass (A/B) */
static bool rb_fold_enabled() { const char *e = getenv("MSQG_RB_FOLD"); return !(e && atoi(e) == 0); }
/* nrelax sweeps on da / res of level l: the layer-coupled problem (mode < 0), or vertical mode `mode` with its lambda
 * (per-cell tables while the modes vary horizontally).  halo, corr_a: launch_relax's */
static int relax_level(msqg_model *m, int mode, int l, int nrelax, int halo = 0, double *corr_a = nullptr) {
  int rc;
  if (mode < 0) {
    NL_SWITCH(m->nl, { auto C = relax_coef_layers<NL>(m, l); rc = launch_relax<NL>(m, m->da.lev[l], m->res.lev[l], l, nrelax, C, halo, corr_a); });
  } else {
    auto C = relax_coef_scalar(m, l, m->lam_lev[(size_t)l * m->nl + mode]);
    m->coef_mode = m->modes_uniform ? -1 : mode;
    rc = launch_relax<1>(m, m->da.lev[l], m->res.lev[l], l, nrelax, C, halo, corr_a);
    m->coef_mode = -1;
  }
  return rc;
}
/* corrected != NULL (mg_cycle): when level D of an undecomposed grid goes through the streaming red-black kernel, its
 * last pass adds da to corr_a (no k_correct); *corrected tells the caller whether that happened.  Same bits. */
static int mg_levels(msqg_model *m, int nf, int mode, int nrelax, int from, int top, double *corr_a = nullptr,
                     bool *corrected = nullptr) {
  dim3 b(32, 8);
  const int D = m->depth;
  const bool fold = corrected && m->smoother == 1 && !m->periodic && rb_fold_enabled();
  if (corrected) *corrected = false;
  const int Lc = coarse_top_level(m, nf, top < D ? top : D - 1);
  /* k_prolong4 and the level relax kernels meet dirichlet ghosts on an undecomposed level: with periodic boundaries every
     level of this loop must be inside the wrap-around coarse kernel (create_model sizes agg_n for that) */
  if (m->periodic && Lc < top) FAIL(MSQG_ERR_ARG, "periodic level %d is not covered by the wrap-around coarse kernel (levels 1 .. %d)", top, Lc);
  for (int l = from - 1; l >= (Lc ? Lc : 1); l--) {
    ProfScope ps(m, PROF_RESTRICT, l);
    k_restrict<<<grid2(m->g[l].nx, m->g[l].ny, b, nf), b, 0, m->stream>>>(m->res.lev[l + 1], m->res.lev[l], m->g[l + 1], m->g[l], -1., 0);
    m->launches++;
  }
  CK(cudaGetLastError());
  int rc = MSQG_OK;
  if (Lc) {
    ProfScope ps(m, PROF_RELAX_COARSE, nrelax);
    if (mode < 0) {
      NL_SWITCH(m->nl, {
        CoarseCoef<NL> CC;
        for (int l = 1; l <= Lc; l++) CC.c[l] = relax_coef_layers<NL>(m, l);
        CC.c[0] = CC.c[1];
        if (relax_uses_table<NL>(m)) {
          if constexpr (NL <= 6) rc = launch_coarse_rb<NL, true>(m, Lc, nrelax, CC);
          else rc = MSQG_ERR_ARG;
        } else
          rc = launch_coarse_rb<NL>(m, Lc, nrelax, CC);
      });
    } else {
      CoarseCoef<1> CC;
      for (int l = 1; l <= Lc; l++) CC.c[l] = relax_coef_scalar(m, l, m->lam_lev[(size_t)l * m->nl + mode]);
      CC.c[0] = CC.c[1];
      m->coef_mode = m->modes_uniform ? -1 : mode;
      rc = m->coef_mode >= 0 ? launch_coarse_rb<1, true>(m, Lc, nrelax, CC) : launch_coarse_rb<1>(m, Lc, nrelax, CC);
      m->coef_mode = -1;
    }
    if (rc) return rc;
  }
  const int minlevel = top < 1 ? top : 1;
  for (int l = Lc ? Lc + 1 : minlevel; l <= top; l++) {
    const Geom &g = m->g[l];
    const bool rcoef = mode < 0 ? !m->s_uniform : !m->modes_uniform; /* relax_uses_table of the launches below */
    double *ca = (fold && l == D && rb_can_fold(nf) && g.bc == 0 && !rb_tiled(nf, rcoef, (long long)g.nx * g.ny)) ? corr_a : nullptr;
    if (l == minlevel) { /* da = 0 on the coarsest level */
      CK(cudaMemsetAsync(m->da.lev[l], 0, (size_t)nf * g.plane * sizeof(double), m->stream));
    } else {
      ProfScope ps(m, PROF_PROLONG, l);
      launch_prolong(m->stream, nf, m->da.lev[l - 1], m->da.lev[l], m->g[l - 1], g);
      m->launches++;
      CK(cudaGetLastError());
    }
    ProfScope ps(m, l == D ? PROF_RELAX_FINE : PROF_RELAX_COARSE, nrelax);
    if ((rc = relax_level(m, mode, l, nrelax, 0, ca))) return rc;
    if (ca) *corrected = true;
  }
  return MSQG_OK;
}

/* mg_cycle, mspg/elliptic.h:43-99 with minlevel = 1 (poisson_layer.h:297) */
static int mg_cycle(msqg_model *m, const MgProblem &P, int nrelax) {
  const int D = m->depth;
  dim3 b(32, 8);
  /* restriction(res): levels D-1..1 (level 0 is never read with minlevel = 1), then levels 1 .. D.  The residual
     before the cycle has already restricted res down to residual_pyr_bottom */
  bool corrected = false;
  int rc = mg_levels(m, P.nf, P.mode, nrelax, residual_pyr_bottom(m), D, P.a, &corrected);
  if (rc) return rc;
  if (corrected) return MSQG_OK; /* corrected: the last relax pass on level D did a += da */
  const Geom &g = m->g[D];
  { ProfScope ps(m, PROF_CORRECT, 0);
  k_correct<<<grid2(g.nx, g.ny, b, P.nf), b, 0, m->stream>>>(P.a, m->da.lev[D], g); }
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* The solve loop of mg_solve and g_solve, mspg/elliptic.h:145-229: NITERMIN=1, NITERMAX=100, nrelax starts at 4 and
 * adapts to the convergence rate.  sched != NULL (msqg_test_cycles): exactly ncycles cycles, cycle k with sched[k]
 * sweeps per level, no tolerance stop and no adaptation; resa_out[k] is the residual after cycle k.
 * residual() and cycle(nrelax) only enqueue work on `st`; read(&r) waits for the residual norm.  Each cycle and the
 * residual that follows it run through run_graphed (one graph launch when `graphed`), keyed by nrelax, the problem
 * (mode, unknown and right-hand side of P, the first tile's under a group) and the da buffers of every model. */
template <class Residual, class Cycle, class Read>
static int mg_solve_loop(cudaStream_t st, GraphCache &gc, std::vector<msqg_model *> &models, long *exchanges, bool graphed,
                         const MgProblem &P, double tolerance, msqg_mgstats *out, const int *sched, int ncycles,
                         double *resa_out, Residual residual, Cycle cycle, Read read) {
  msqg_mgstats s;
  memset(&s, 0, sizeof(s));
  s.nrelax = 4;
  double resb;
  int rc;
  if ((rc = residual()) || (rc = read(&resb))) return rc;
  s.resb = s.resa = resb;
  for (s.i = 0; sched ? s.i < ncycles : s.i < 100 && (s.i < 1 || s.resa > tolerance); s.i++) {
    if (sched) s.nrelax = sched[s.i];
    unsigned long long mask = 0;
    for (msqg_model *m : models) mask = mask * 1315423911ull + da_parity_mask(m);
    GraphKey key(s.nrelax, P.mode, (const void *)P.a, (const void *)P.b, mask);
    rc = run_graphed(st, gc, key, models, exchanges, graphed, [&]() -> int {
      int r2 = cycle(s.nrelax);
      if (r2) return r2;
      return residual();
    });
    if (rc || (rc = read(&s.resa))) return rc;
    if (sched) resa_out[s.i] = s.resa;
    else if (s.resa > tolerance) {
      if (resb / s.resa < 1.2 && s.nrelax < 100) s.nrelax++;
      else if (resb / s.resa > 10 && s.nrelax > 2) s.nrelax--;
    }
    resb = s.resa;
  }
  *out = s;
  return MSQG_OK;
}

/* mg_solve on one grid; sched, ncycles, resa_out as mg_solve_loop's */
static int mg_solve(msqg_model *m, const MgProblem &P, double tolerance, msqg_mgstats *st, const int *sched = nullptr,
                    int ncycles = 0, double *resa_out = nullptr) {
  const bool graphed = m->smoother == 1 && m->use_graphs && !m->prof_on; /* coefficient tables are fixed between set_const calls */
  std::vector<msqg_model *> self(1, m);
  msqg_mgstats s;
  int rc = mg_solve_loop(m->stream, m->graphs, self, nullptr, graphed, P, tolerance, &s, sched, ncycles, resa_out,
                         [&]() { return mg_residual_enqueue(m, P); },
                         [&](int nrelax) { return mg_cycle(m, P, nrelax); },
                         [&](double *r) { return mg_residual_read(m, r); });
  if (rc || (rc = check_relax_err(m))) return rc;
  m->total_cycles += s.i;
  *st = s;
  return MSQG_OK;
}

/* layers <-> vertical modes on level D (k_project): out = M in with the host matrix h_mat, or with the per-column
 * matrices of the field matf (non-null: horizontally varying modes).  ring: also the one-cell ring of a tile;
 * ghosts: k_project's last argument */
static int launch_project(msqg_model *m, const double *in, double *out, const double *h_mat, const double *matf, bool ring,
                          int ghosts) {
  const Geom &g = m->g[m->depth];
  dim3 b(64, 4);
  NL_SWITCH(m->nl, {
    ModeMat<NL> M;
    for (int k = 0; k < NL * NL; k++) M.a[k] = h_mat[k];
    if (ring) k_project<NL, true><<<grid2(g.nx + 2, g.ny + 2, b), b, 0, m->stream>>>(in, out, g, M, matf, ghosts);
    else k_project<NL><<<grid2(g.nx, g.ny, b), b, 0, m->stream>>>(in, out, g, M, matf, ghosts);
  });
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* invertq, msqg/qg.h:113-163 */
static int invertq_list(msqg_model *m, List &ql) {
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "set_const must be called before invertq");
  const int D = m->depth;
  const Geom &g = m->g[D];
  int rc;
  if (!m->p.mode_pv_invert) {
    MgProblem P{m->nl, -1, m->psi.lev[D], ql.lev[D]};
    if ((rc = mg_solve(m, P, 1e-3, &m->mgpsi))) return rc;
  } else {
    /* horizontally varying Fr/Ro: the projection matrices are fields (one eigmod per column), as in the reference */
    const double *matf_l2m = m->modes_uniform ? nullptr : m->cl2m.lev[D];
    const double *matf_m2l = m->modes_uniform ? nullptr : m->cm2l.lev[D];
    if ((rc = launch_project(m, ql.lev[D], m->qm.lev[D], m->h_cl2m, matf_l2m, false, 0))) return rc;
    for (int l = 0; l < m->nl; l++) {
      MgProblem P{1, l, m->pm.lev[D] + (size_t)l * g.plane, m->qm.lev[D] + (size_t)l * g.plane};
      if ((rc = mg_solve(m, P, 1e-3, &m->mgmode[l]))) return rc;
      m->mgpsi = m->mgmode[l];
    }
    if ((rc = launch_project(m, m->pm.lev[D], m->psi.lev[D], m->h_cm2l, matf_m2l, false, 1))) return rc;
  }
  return MSQG_OK;
}
extern "C" int msqg_invertq(msqg_model *m, int q_id) {
  CK(cudaSetDevice(m->device));
  List *L = list_by_id(m, q_id);
  if (!L || L->nf != m->nl) FAIL(MSQG_ERR_ARG, "bad q list");
  if (m->group) return pg_invertq(m->group, m, q_id);
  return invertq_list(m, *L);
}

extern "C" int msqg_comp_q(msqg_model *m) {
  CK(cudaSetDevice(m->device));
  if (m->group) { int rc = pg_halo(m->group, MSQG_PSI); if (rc) return rc; } /* psi across the seam */
  const Geom &g = m->g[m->depth];
  dim3 b(64, 4);
  LayerMetrics M = metrics_of(m);
  NL_SWITCH(m->nl, k_comp_q<NL><<<grid2(g.nx, g.ny, b), b, 0, m->stream>>>(m->psi.lev[m->depth], m->str.lev[m->depth], m->q.lev[m->depth], g, M));
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* ------------------------------------------------------------------ eigmod (setup) */
typedef void (*dgeev_fn)(const char *, const char *, const int *, double *, const int *, double *, double *, double *,
                         const int *, double *, const int *, double *, const int *, int *, size_t, size_t);
static dgeev_fn find_dgeev() {
  static dgeev_fn fn = nullptr;
  static bool tried = false;
  if (tried) return fn;
  tried = true;
  const char *cands[] = {getenv("MSQG_LAPACK"), "liblapack.so.3", "liblapack.so", "libopenblas.so.0", "libopenblas.so"};
  for (const char *c : cands) {
    if (!c) continue;
    void *h = dlopen(c, RTLD_NOW | RTLD_GLOBAL);
    if (!h) continue;
    fn = (dgeev_fn)dlsym(h, "dgeev_");
    if (!fn) fn = (dgeev_fn)dlsym(h, "scipy_dgeev_");
    if (fn) break;
  }
  return fn;
}
struct eig_pair { double v; int idx; };
static int cmp_eig(const void *a, const void *b) {
  double x = ((const eig_pair *)a)->v, y = ((const eig_pair *)b)->v;
  return (x > y) - (x < y);
}
/* eigmod for one column, msqg/eigmode.h:74-266 (LAPACKE_dgeev row-major == dgeev_
 * on the transposed matrix with vl/vr transposed back) */
static int eigmod_column(int nl, const double *dhf, const double *Fr, double Ro, double *cl2m, double *cm2l, double *iBu) {
  dgeev_fn dgeev = find_dgeev();
  if (!dgeev) FAIL(MSQG_ERR_CONFIG, "MODE_PV_INVERT needs LAPACK dgeev (msqg/eigmode.h:153): set MSQG_LAPACK to a LAPACK/OpenBLAS shared library");
  double dhc[MSQG_MAXL];
  for (int l = 0; l < nl - 1; l++) dhc[l] = 0.5 * (dhf[l] + dhf[l + 1]);
  std::vector<double> amat((size_t)nl * nl, 0.), acm((size_t)nl * nl), vl((size_t)nl * nl), vr((size_t)nl * nl),
      vlc((size_t)nl * nl), vrc((size_t)nl * nl), tmp((size_t)nl * nl);
  double wr[MSQG_MAXL], wi[MSQG_MAXL];
  eig_pair wr2[MSQG_MAXL];
  {
    int l = 0;
    amat[nl * l + l + 1] = -sq(Fr[l] / Ro) / (dhc[l] * dhf[l]);
    amat[nl * l + l] = -amat[nl * l + l + 1];
    for (l = 1; l < nl - 1; l++) {
      amat[nl * l + l - 1] = -sq(Fr[l - 1] / Ro) / (dhc[l - 1] * dhf[l]);
      amat[nl * l + l + 1] = -sq(Fr[l] / Ro) / (dhc[l] * dhf[l]);
      amat[nl * l + l] = -amat[nl * l + l - 1] - amat[nl * l + l + 1];
    }
    l = nl - 1;
    amat[nl * l + l - 1] = -sq(Fr[l - 1] / Ro) / (dhc[l - 1] * dhf[l]);
    amat[nl * l + l] = -amat[nl * l + l - 1];
  }
  for (int r = 0; r < nl; r++)
    for (int c = 0; c < nl; c++) acm[r + nl * c] = amat[nl * r + c];
  int info = 0, lwork = 8 * nl + 64;
  std::vector<double> work(lwork);
  dgeev("V", "V", &nl, acm.data(), &nl, wr, wi, vlc.data(), &nl, vrc.data(), &nl, work.data(), &lwork, &info, 1, 1);
  if (info < 0) FAIL(MSQG_ERR_CONFIG, "issue with lapack in eigmode (info=%d)", info);
  for (int r = 0; r < nl; r++)
    for (int c = 0; c < nl; c++) { vl[r * nl + c] = vlc[r + nl * c]; vr[r * nl + c] = vrc[r + nl * c]; }
  for (int l = 0; l < nl; l++) { wr2[l].v = wr[l]; wr2[l].idx = l; }
  qsort(wr2, nl, sizeof(eig_pair), cmp_eig);
  for (int l = 0; l < nl; l++) wr[l] = wr2[l].v;
  tmp = vr;
  for (int mm = 0; mm < nl; mm++)
    for (int k = 0; k < nl; k++) vr[k * nl + mm] = tmp[k * nl + wr2[mm].idx];
  tmp = vl;
  for (int mm = 0; mm < nl; mm++)
    for (int k = 0; k < nl; k++) vl[k * nl + mm] = tmp[k * nl + wr2[mm].idx];
  const double htotal = 1.;
  for (int mm = 0; mm < nl; mm++) {
    double dotp = 0.;
    for (int k = 0; k < nl; k++) dotp += dhf[k] * vr[k * nl + mm] * vr[k * nl + mm];
    const double flfac = (vr[mm] > 0 ? 1 : -1) * sqrt(htotal / dotp);
    for (int k = 0; k < nl; k++) vr[k * nl + mm] = flfac * vr[k * nl + mm];
  }
  for (int mm = 0; mm < nl; mm++) {
    double dotp = 0.;
    for (int k = 0; k < nl; k++) dotp += vr[k * nl + mm] * vl[k * nl + mm];
    for (int k = 0; k < nl; k++) vl[k * nl + mm] = vl[k * nl + mm] / dotp;
  }
  for (int mm = 0; mm < nl; mm++)
    for (int k = 0; k < nl; k++) {
      cl2m[k * nl + mm] = vl[mm * nl + k];
      cm2l[k * nl + mm] = vr[k * nl + mm];
    }
  for (int l = 0; l < nl; l++) iBu[l] = -wr[l];
  iBu[0] = 0.;
  return MSQG_OK;
}

/* ------------------------------------------------------------------ set_const */
static inline double avg4(double a, double b, double c, double d) {
  /* [BASILISK] restriction_average order */
  double sum = 0.;
  sum += a; sum += b; sum += c; sum += d;
  return sum / 4;
}

static int max_face_speed(msqg_model *m, List &L, double *umax_host) {
  const int D = m->depth;
  const Geom &g = m->g[D];
  CK(zero_words(m->stream, m->d_scal + 1, m->nl));
  dim3 b(64, 4);
  /* out-of-place laplacian into tmp is a by-product; only umax is wanted */
  launch_lap(m->stream, m->nl, L.lev[D], m->tmp.lev[D], g, m->d_scal + 1, m->sbcc);
  m->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(m->h_scal + 1, m->d_scal + 1, m->nl * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  for (int l = 0; l < m->nl; l++) umax_host[l] = m->h_scal[1 + l];
  return MSQG_OK;
}

/* varRo > 0: the stretching depends on y only -> per-row Thomas coefficients for the relax kernel, built on the device
 * from the restricted stretching field of levels lo .. hi (same expressions as relax_coef_layers); stretching that varies
 * with x as well (Fr from frpg_*.bas, qg.h:957-962): the same table per CELL.  On the levels of a tile the table also
 * covers the halo of the internal sides, as deep as the sweeps of one exchange reach (g_cycle: at most MSQG_FRAME - 1
 * cells, capped at the tile size); the stretching must have been exchanged there. */
static int build_stretch_tables(msqg_model *m, int lo, int hi) {
  const int nl = m->nl;
  const LayerMetrics M = metrics_of(m);
  const int cell = m->s_rowuniform ? 0 : 1;
  for (int l = lo; l <= hi; l++) {
    const Geom &gl = m->g[l];
    if (m->rowcoef[l]) { CK(cudaFree(m->rowcoef[l])); m->rowcoef[l] = nullptr; }
    int mg = MSQG_FRAME - 1;
    if (mg > gl.nx) mg = gl.nx;
    if (mg > gl.ny) mg = gl.ny;
    const int mx = (gl.bc & 1) ? mg : 0, my = (gl.bc & 4) ? mg : 0;
    const int tw = gl.nx + mx + ((gl.bc & 2) ? mg : 0), th = gl.ny + my + ((gl.bc & 8) ? mg : 0);
    m->coef_mx[l] = mx; m->coef_my[l] = my; m->coef_w[l] = tw;
    const size_t ent = (size_t)th * (cell ? tw : 1);
    CK(cudaMalloc(&m->rowcoef[l], ent * 6 * nl * sizeof(double)));
    NL_SWITCH(nl, k_rowcoef<NL><<<(unsigned)((ent + 127) / 128), 128, 0, m->stream>>>(m->str.lev[l], gl, M, m->rowcoef[l], cell, -mx, -my, tw, th));
    m->launches++;
  }
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* set_const up to (not including) comp_q: everything that is local to a tile.  tables = false (tiles of a group): no
 * stretching tables, the group builds them once it has decided the path for all tiles */
static int set_const_local(msqg_model *m, bool tables = true) {
  CK(cudaSetDevice(m->device));
  m->graphs.clear(); /* recorded cycles hold the old coefficients */
  const int nl = m->nl, D = m->depth;
  const int tx = m->tnx, ty = m->tny; /* finest tile (whole grid on one GPU) */
  const size_t tc = (size_t)tx * ty;
  const double Delta = m->p.L0 / m->N;
  /* sanity checks, qg.h:990-1012 */
  for (int l = 0; l < nl; l++)
    if (m->dhf[l] == 0) FAIL(MSQG_ERR_CONFIG, "thickness = 0: aborting\nCheck the definition of dh in params.in");
  if (m->p.Rom <= 0) FAIL(MSQG_ERR_CONFIG, "Rom <= 0: aborting");
  /* layer metrics, qg.h:1017-1027 */
  for (int l = 0; l < nl - 1; l++) m->dhc[l] = 0.5 * (m->dhf[l] + m->dhf[l + 1]);
  m->idh0[0] = 0.;
  m->idh1[0] = 1. / (m->dhc[0] * m->dhf[0]);
  for (int l = 1; l < nl - 1; l++) {
    m->idh0[l] = 1. / (m->dhc[l - 1] * m->dhf[l]);
    m->idh1[l] = 1. / (m->dhc[l] * m->dhf[l]);
  }
  m->idh0[nl - 1] = 1. / (m->dhc[nl - 2] * m->dhf[nl - 1]);
  m->idh1[nl - 1] = 0.;
  /* Ro(y), qg.h:1032-1037 */
  std::vector<double> ro_y(ty);
  for (int j = 0; j < ty; j++) {
    const double y = (m->y0 + j + 0.5) * Delta;
    ro_y[j] = m->p.varRo > 0 ? m->p.Rom / (1 + m->p.Rom * m->p.beta * (y - 0.5 * m->p.L0)) : m->p.Rom;
  }
  int rc;
  {
    std::vector<double> h(tc);
    for (int j = 0; j < ty; j++)
      for (int i = 0; i < tx; i++) h[(size_t)j * tx + i] = ro_y[j];
    if ((rc = pack_to(m, m->ro, h.data()))) return rc;
  }
  /* strl = sq(Fr/Ro), qg.h:1043-1048 (layers 0..nl-2; layer nl-1 stays 0) */
  std::vector<double> hs((size_t)nl * tc, 0.);
  bool uniform = true, rowuniform = true;
  for (int l = 0; l < nl - 1; l++) {
    const double *fr = &m->h_fr[(size_t)l * tc];
    double *s = &hs[(size_t)l * tc];
    for (int j = 0; j < ty; j++)
      for (int i = 0; i < tx; i++) s[(size_t)j * tx + i] = sq(fr[(size_t)j * tx + i] / ro_y[j]);
    for (size_t c = 1; c < tc && uniform; c++) uniform = s[c] == s[0];
    for (int j = 0; j < ty && rowuniform; j++)
      for (int i = 1; i < tx && rowuniform; i++) rowuniform = s[(size_t)j * tx + i] == s[(size_t)j * tx];
  }
  if ((rc = pack_to(m, m->str, hs.data()))) return rc;
  m->s_uniform = uniform;
  m->s_rowuniform = rowuniform;
  /* restriction(strl) (poisson_layer.h:284): fields on the device, per-level
     constants on the host for the uniform case (same summation order) */
  {
    dim3 b(32, 8);
    /* tiles restrict only their distributed levels: coarser-level stretching enters the kernels
       through the per-level constants s_lev (uniform stretching) */
    for (int l = D - 1; l >= (m->agg_level > 1 ? m->agg_level : 1); l--) {
      k_restrict<<<grid2(m->g[l].nx, m->g[l].ny, b, nl), b, 0, m->stream>>>(m->str.lev[l + 1], m->str.lev[l], m->g[l + 1], m->g[l], 1., 1);
      m->launches++;
    }
    CK(cudaGetLastError());
  }
  m->s_lev.assign((size_t)(D + 1) * nl, 0.);
  if (uniform) {
    for (int l = 0; l < nl - 1; l++) m->s_lev[(size_t)D * nl + l] = hs[(size_t)l * tc];
    for (int lev = D - 1; lev >= 0; lev--)
      for (int l = 0; l < nl; l++) {
        const double v = m->s_lev[(size_t)(lev + 1) * nl + l];
        m->s_lev[(size_t)lev * nl + l] = avg4(v, v, v, v);
      }
  }
  for (int l = 0; l <= MSQG_MAXLEV; l++) if (m->rowcoef[l]) { CK(cudaFree(m->rowcoef[l])); m->rowcoef[l] = nullptr; }
  /* a group decides uniform / per-row / per-cell for all its tiles together and builds their tables itself (g_stretching) */
  if (tables && !uniform && (rc = build_stretch_tables(m, 1, D))) return rc;
  /* wind forcing table, qg.h:451, host libm so that sin() matches the reference */
  {
    std::vector<double> w(ty);
    const double pi = 3.14159265358979323846, L0 = m->p.L0;
    for (int j = 0; j < ty; j++) {
      const double y = (m->y0 + j + 0.5) * Delta;
      w[j] = m->p.tau0 / (m->p.Rom * m->dhf[0]) * sin(2 * pi * y / L0) * sin(pi * y / L0);
    }
    CK(cudaMemcpyAsync(m->d_wind, w.data(), ty * sizeof(double), cudaMemcpyHostToDevice, m->stream));
    CK(cudaStreamSynchronize(m->stream));
  }
  std::vector<double> sig(tc);
  if (m->p.mode_pv_invert) {
    /* eigmod, qg.h:1053 -> eigmode.h:65-308.  Inputs depend on (Fr, Ro) only. */
    bool fr_uniform = true;
    for (int l = 0; l < nl - 1 && fr_uniform; l++)
      for (size_t c = 1; c < tc && fr_uniform; c++) fr_uniform = m->h_fr[(size_t)l * tc + c] == m->h_fr[(size_t)l * tc];
    m->modes_uniform = fr_uniform && m->p.varRo <= 0;
    for (int k = 0; k < MSQG_NLMAX; k++)
      for (int l = 0; l <= MSQG_MAXLEV; l++) if (m->modecoef[k][l]) { CK(cudaFree(m->modecoef[k][l])); m->modecoef[k][l] = nullptr; }
    m->lam_lev.assign((size_t)(D + 1) * nl, 0.);
    if (m->modes_uniform) {
      double fr[MSQG_MAXL];
      for (int l = 0; l < nl - 1; l++) fr[l] = m->h_fr[(size_t)l * tc];
      if ((rc = eigmod_column(nl, m->dhf, fr, ro_y[0], m->h_cl2m, m->h_cm2l, m->h_ibu))) return rc;
      std::vector<double> h((size_t)nl * nl * tc);
      for (int k = 0; k < nl * nl; k++) for (size_t c = 0; c < tc; c++) h[(size_t)k * tc + c] = m->h_cl2m[k];
      if ((rc = pack_to(m, m->cl2m, h.data()))) return rc;
      for (int k = 0; k < nl * nl; k++) for (size_t c = 0; c < tc; c++) h[(size_t)k * tc + c] = m->h_cm2l[k];
      if ((rc = pack_to(m, m->cm2l, h.data()))) return rc;
      for (int k = 0; k < nl; k++) for (size_t c = 0; c < tc; c++) h[(size_t)k * tc + c] = m->h_ibu[k];
      if ((rc = pack_to(m, m->ibu, h.data()))) return rc;
      /* poisson(): restriction({alpha,lambda}) [BASILISK] -> per-level lambda */
      for (int l = 0; l < nl; l++) m->lam_lev[(size_t)D * nl + l] = m->h_ibu[l];
      for (int lev = D - 1; lev >= 0; lev--)
        for (int l = 0; l < nl; l++) {
          const double v = m->lam_lev[(size_t)(lev + 1) * nl + l];
          m->lam_lev[(size_t)lev * nl + l] = avg4(v, v, v, v);
        }
      for (size_t c = 0; c < tc; c++) sig[c] = fmin(m->p.afilt * sqrt(-1 / m->h_ibu[1]), m->p.Lfmax);
    } else {
      /* one dgeev per column, as the reference does (eigmode.h:74-299).  LAPACK is deterministic, so columns with the
         inputs of the previous one (every column of a row when only Ro(y) varies) reuse its result. */
      if (m->g[D].bc || m->agg_level > 1) FAIL(MSQG_ERR_ARG, "MODE_PV_INVERT with spatially varying Fr/Ro is not supported on decomposed grids");
      std::vector<double> hl((size_t)nl * nl * tc), hm((size_t)nl * nl * tc), hb((size_t)nl * tc);
      double cl[MSQG_NLMAX * MSQG_NLMAX], cm[MSQG_NLMAX * MSQG_NLMAX], ib[MSQG_NLMAX], fr[MSQG_MAXL], last_fr[MSQG_MAXL], last_ro = 0.;
      bool have = false;
      for (int j = 0; j < ty; j++)
        for (int i = 0; i < tx; i++) {
          const size_t c = (size_t)j * tx + i;
          for (int l = 0; l < nl - 1; l++) fr[l] = m->h_fr[(size_t)l * tc + c];
          bool same = have && ro_y[j] == last_ro;
          for (int l = 0; same && l < nl - 1; l++) same = fr[l] == last_fr[l];
          if (!same) {
            if ((rc = eigmod_column(nl, m->dhf, fr, ro_y[j], cl, cm, ib))) return rc;
            have = true; last_ro = ro_y[j];
            for (int l = 0; l < nl - 1; l++) last_fr[l] = fr[l];
          }
          for (int k = 0; k < nl * nl; k++) { hl[(size_t)k * tc + c] = cl[k]; hm[(size_t)k * tc + c] = cm[k]; }
          for (int k = 0; k < nl; k++) hb[(size_t)k * tc + c] = ib[k];
          sig[c] = fmin(m->p.afilt * sqrt(-1 / ib[1]), m->p.Lfmax);
        }
      for (int k = 0; k < nl * nl; k++) { m->h_cl2m[k] = hl[(size_t)k * tc]; m->h_cm2l[k] = hm[(size_t)k * tc]; }
      for (int k = 0; k < nl; k++) m->h_ibu[k] = hb[(size_t)k * tc];
      if ((rc = pack_to(m, m->cl2m, hl.data()))) return rc;
      if ((rc = pack_to(m, m->cm2l, hm.data()))) return rc;
      if ((rc = pack_to(m, m->ibu, hb.data()))) return rc;
      /* poisson(): restriction({alpha, lambda}) [BASILISK], then the relax tables of every mode and level */
      dim3 b(32, 8);
      for (int l = D - 1; l >= 1; l--) {
        k_restrict<<<grid2(m->g[l].nx, m->g[l].ny, b, nl), b, 0, m->stream>>>(m->ibu.lev[l + 1], m->ibu.lev[l], m->g[l + 1], m->g[l], 1., 1);
        m->launches++;
      }
      CK(cudaGetLastError());
      for (int k = 0; k < nl; k++)
        for (int l = 1; l <= D; l++) {
          const Geom &gl = m->g[l];
          const size_t ent = (size_t)gl.ny * gl.nx;
          CK(cudaMalloc(&m->modecoef[k][l], ent * 6 * sizeof(double)));
          k_modecoef<<<(unsigned)((ent + 127) / 128), 128, 0, m->stream>>>(m->ibu.lev[l] + (size_t)k * gl.plane, gl, m->modecoef[k][l]);
          m->launches++;
        }
      CK(cudaGetLastError());
    }
  } else {
    std::vector<double> rd(tc);
    if ((rc = unpack_from(m, m->rd, rd.data()))) return rc;
    for (size_t c = 0; c < tc; c++) sig[c] = fmin(m->p.afilt * rd[c], m->p.Lfmax);
  }
  if ((rc = pack_to(m, m->sigfilt, sig.data()))) return rc;
  m->h_sigfilt = sig;
  m->filter_vars = 0; /* sig_lev is rebuilt from the new sig_filt on the next filter call */
  m->const_set = 1;
  return MSQG_OK;
}

/* the rest of set_const: needs psi / psi_pg ghosts (already consistent on one GPU) */
static int set_const_finish(msqg_model *m) {
  const int nl = m->nl, D = m->depth;
  const Geom &g = m->g[D];
  int rc;
  /* comp_q(pol,qol), qg.h:1092 */
  if ((rc = msqg_comp_q(m))) return rc;
  /* flsrv: zeta_pg = laplacian(psi_pg), qg.h:1094-1097; also its CFL speeds (static) */
  m->has_zp = 0;
  if (m->has_pg) {
    if ((rc = max_face_speed(m, m->psipg, m->umax_pg))) return rc;
    if (m->p.flsrv == 1) {
      dim3 b(64, 4);
      /* set_const ends with boundary(all) (qg.h:1103), which puts the dirichlet ghosts back on zetapl after the
         partial-slip fix-up of comp_del2: sbcc = 0 here */
      launch_lap(m->stream, nl, m->psipg.lev[D], m->zetap.lev[D], g, nullptr, 0.);
      m->launches++;
      CK(cudaGetLastError());
      m->has_zp = 1;
    }
  } else
    for (int l = 0; l < nl; l++) m->umax_pg[l] = 0.;
  CK(cudaStreamSynchronize(m->stream));
  return MSQG_OK;
}

extern "C" int msqg_set_const(msqg_model *m) {
  if (m->group) return pg_set_const(m->group);
  int rc = set_const_local(m);
  if (rc) return rc;
  return set_const_finish(m);
}

/* ------------------------------------------------------------------ RHS */
/* timestep() [BASILISK] given the max face speed of one face vector */
static double timestep_chain(msqg_model *m, double umax, double dtmax, double Delta) {
  const double CFL = m->p.CFL;
  dtmax /= CFL;
  if (umax != 0.) {
    const double dt = Delta / umax;
    if (dt < dtmax) dtmax = dt;
  }
  dtmax *= CFL;
  if (dtmax > m->ts_previous) dtmax = (m->ts_previous + 0.1 * dtmax) / 1.1;
  m->ts_previous = dtmax;
  return dtmax;
}

/* zeta = laplacian(psi) (+ umax), tmp = laplacian(zeta) if viscosity is on */
static int rhs_prepare(msqg_model *m) {
  const int D = m->depth;
  const Geom &g = m->g[D];
  dim3 b(64, 4);
  CK(zero_words(m->stream, m->d_scal + 1, m->nl));
  ProfScope ps(m, PROF_LAP, 0);
  launch_lap(m->stream, m->nl, m->psi.lev[D], m->zeta.lev[D], g, m->d_scal + 1, m->sbcc);
  m->launches++;
  if (m->iRe != 0. || m->iRe4 != 0.) {
    launch_lap(m->stream, m->nl, m->zeta.lev[D], m->tmp.lev[D], g, nullptr, m->sbcc);
    m->launches++;
  }
  CK(cudaGetLastError());
  CK(to_host(m->stream, m->h_scal + 1, m->d_scal + 1, m->nl));
  return MSQG_OK;
}
/* dtmax chain of advection_pv, qg.h:383-391: umax, the max face speeds of psi (needs their D2H to have completed), and
 * umax_pg, those of the background flow, per layer.  timestep()'s state is m->ts_previous (a group's: its tiles[0]'s) */
static double dt_chain(msqg_model *m, const double *umax, const double *umax_pg, double dtmax) {
  const double Delta = m->g[m->depth].Delta;
  for (int l = 0; l < m->nl; l++) {
    dtmax = timestep_chain(m, umax[l], dtmax, Delta);
    dtmax = timestep_chain(m, umax_pg[l], dtmax, Delta);
  }
  return dtmax;
}
/* dtnext(), [BASILISK] events: TEPS = 1e-9.  dt rounded so that t lands on tnext_event (negative: no pending event);
 * *tnext is the time after the step */
static double dtnext(double t, double tnext_event, double dt, double *tnext) {
  if (tnext_event >= 0 && tnext_event > t) {
    unsigned int nn = (tnext_event - t) / dt;
    *tnext = tnext_event;
    if (nn == 0) dt = tnext_event - t;
    else {
      const double dt1 = (tnext_event - t) / nn;
      if (dt1 > dt * (1. + 1e-9)) dt = (tnext_event - t) / (nn + 1);
      else if (dt1 < dt) dt = dt1;
      *tnext = t + dt;
    }
  } else
    *tnext = t + dt;
  return dt;
}

static int rhs_launch(msqg_model *m, List &q_ev, const double *q_in, double *q_out, double *dq, double dt, float dts) {
  const int D = m->depth;
  const Geom &g = m->g[D];
  const int nl = m->nl;
  RhsArgs A;
  memset(&A, 0, sizeof(A));
  A.psi = m->psi.lev[D]; A.zeta = m->zeta.lev[D]; A.tmp = m->tmp.lev[D]; A.pp = m->psipg.lev[D];
  A.zp = m->zetap.lev[D]; A.s = m->str.lev[D]; A.qforc = m->has_qforc ? m->qforc.lev[D] : nullptr;
  A.topo = m->topo.lev[D]; A.ro = m->ro.lev[D];
  A.q_in = q_in; A.q_ev = q_ev.lev[D]; A.q_out = q_out; A.dq = dq;
  A.noise = m->p.stochastic ? m->nstoch.lev[D] : nullptr;
  A.wind = m->d_wind; A.g = g;
  for (int l = 0; l < nl; l++) { A.idh0[l] = m->idh0[l]; A.idh1[l] = m->idh1[l]; }
  A.beta = m->p.beta; A.iRe = m->iRe; A.iRe4 = m->iRe4;
  A.ceks = m->Eks / (m->p.Rom * 2 * m->dhf[0]);
  A.cekb = m->Ekb / (m->p.Rom * 2 * m->dhf[nl - 1]);
  A.dhb = m->dhf[nl - 1];
  A.dt = dt; A.itr = m->p.itr_stoch; A.dts = dts;
  A.has_pg = m->has_pg; A.has_zp = m->has_zp; A.use_tmp = (m->iRe != 0. || m->iRe4 != 0.);
  A.flag_topo = m->flag_topo; A.stochastic = m->p.stochastic;
  A.econs = (m->econs && !m->p.stochastic) ? 1 : 0;
  if (A.econs) {
    /* ENERGY_CONSERV (qg.h:310-373): J(psi, q) reads the 3 x 3 neighbourhood of the evolving PV, ghosts included;
       the fused stage update does not keep them (nothing else reads them), so they are rebuilt here */
    if (g.bc) FAIL(MSQG_ERR_ARG, "the ENERGY_CONSERV variant is not available on decomposed grids");
    dim3 bg(32, 8);
    k_ghosts<<<grid2(g.nx + 2, g.ny + 2, bg, nl), bg, 0, m->stream>>>(q_ev.lev[D], nl, g, -1.);
    m->launches++;
  }
  ProfScope ps(m, PROF_RHS, 0);
  static int rhs_variant = -1; /* MSQG_RHS=gather keeps the L1-gather kernel on every configuration (A/B measurements) */
  if (rhs_variant < 0) { const char *e = getenv("MSQG_RHS"); rhs_variant = (e && !strcmp(e, "gather")) ? 0 : 1; }
  if (rhs_variant == 1 && !A.has_pg && !A.has_zp && !A.flag_topo && !A.stochastic && !A.econs) {
    dim3 bt(RT_X, RT_Y);
    NL_SWITCH(nl, k_rhs_t<NL><<<grid2(g.nx, g.ny, bt), bt, 0, m->stream>>>(A));
  } else {
    dim3 b(32, 4);
    NL_SWITCH(nl, k_rhs<NL><<<grid2(g.nx, g.ny, b), b, 0, m->stream>>>(A));
  }
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* ptr_rhs on the tracer tail of `evolving` (qg.h:634-647), optionally fused with the stage update of the tracers */
static int ptr_launch(msqg_model *m, List &tr, const double *tr_in, double *tr_out, double *dptr, double dt) {
  if (m->p.nptr <= 0) return MSQG_OK;
  if (m->g[m->depth].bc) FAIL(MSQG_ERR_ARG, "passive tracers are not supported on decomposed grids");
  const int D = m->depth;
  const Geom &g = m->g[D];
  PtrArgs A;
  memset(&A, 0, sizeof(A));
  A.psi = m->psi.lev[D]; A.ptr = tr.lev[D]; A.relax = m->ptr_relax.lev[D];
  A.ptr_in = tr_in; A.ptr_out = tr_out; A.dptr = dptr; A.g = g; A.dt = dt; A.nptr = m->p.nptr;
  for (int nt = 0; nt < m->p.nptr; nt++) { A.iPe[nt] = m->p.iPe[nt]; A.ptr_ir[nt] = m->p.ptr_ir[nt]; }
  dim3 b(64, 4);
  k_ptr_rhs<<<grid2(g.nx, g.ny, b, tr.nf), b, 0, m->stream>>>(A);
  m->launches++;
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* update_qg(evolving = q_id, updates = DQ, dtmax), qg.h:609-650 */
extern "C" int msqg_update(msqg_model *m, int q_id, double dtmax, double *dtmax_out) {
  CK(cudaSetDevice(m->device));
  List *L = list_by_id(m, q_id);
  if (!L || L->nf != m->nl) FAIL(MSQG_ERR_ARG, "bad q list");
  if (m->group) return pg_update(m->group, m, q_id, dtmax, dtmax_out);
  int rc;
  if ((rc = invertq_list(m, *L))) return rc;
  if ((rc = rhs_prepare(m))) return rc;
  if ((rc = rhs_launch(m, *L, nullptr, nullptr, m->dq.lev[m->depth], 0., 0.f))) return rc;
  if (m->p.nptr > 0 && (rc = ptr_launch(m, q_id == MSQG_QPRED ? m->ptr_pred : m->ptr, nullptr, nullptr, m->dptr.lev[m->depth], 0.))) return rc;
  CK(cudaStreamSynchronize(m->stream));
  if (dtmax_out) *dtmax_out = dt_chain(m, m->h_scal + 1, m->umax_pg, dtmax);
  return MSQG_OK;
}

/* normal_noise / generate_noise, qg_stochastic.h:9,117-126: libc rand() in the
 * reference traversal order (x outer, y inner, layer innermost) on the host.
 * A tile (decomposed or periodic group) replays the WHOLE N x N x nl stream of the undecomposed grid from its own
 * random_r state and keeps the cells of its window [x0, x0 + tnx) x [y0, y0 + tny): the same bits as the
 * undecomposed draw, at O(N^2 nl) host time per draw on every tile (every rank under NCCL).  That is the parity
 * mode; the Philox mode draws only the tile's cells on the device. */
static int generate_noise(msqg_model *m) {
  const int n = m->N, nl = m->nl, tx = m->tnx, ty = m->tny, x0 = m->x0, y0 = m->y0;
  const double pi = 3.14159265358979323846;
  m->noise_draw++;
  if (m->noise_mode == 1) { /* one kernel, no host work: the production mode (and the only one that keeps a GPU busy) */
    const Geom &g = m->g[m->depth];
    dim3 b(64, 4);
    k_noise_philox<<<grid2(g.nx, g.ny, b, nl), b, 0, m->stream>>>(m->nstoch.lev[m->depth], m->sstoch.lev[m->depth], g, n, x0, y0,
                                                                   m->p.amp_stoch, m->noise_seed, m->noise_draw - 1);
    m->launches++;
    CK(cudaGetLastError());
    return MSQG_OK;
  }
  if (m->h_sstoch.empty()) m->h_sstoch.assign((size_t)nl * tx * ty, 0.);
  m->h_noise.resize((size_t)nl * tx * ty);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      const bool mine = i >= x0 && i < x0 + tx && j >= y0 && j < y0 + ty;
      for (int l = 0; l < nl; l++) {
        /* normal_noise(): the two rand() calls in the order gcc evaluates the reference macro's operands */
        int32_t r1, r2;
        random_r(&m->rng, &r1);
        random_r(&m->rng, &r2);
        if (!mine) continue;
        const double gsn = sqrt(-2. * log(((double)(r1) + 1.) / ((double)(RAND_MAX) + 2.))) *
                           cos(2 * pi * r2 / (double)RAND_MAX);
        const size_t c = ((size_t)l * ty + j - y0) * tx + i - x0;
        m->h_noise[c] = m->p.amp_stoch * m->h_sstoch[c] * gsn;
      }
    }
  return pack_to(m, m->nstoch, m->h_noise.data());
}

/* the noise part of one stochastic stage, qg_stochastic.h:128-138: the corrector flag toggles, and every other stage
 * draws a field and scales the noise by 1/sqrt(2); sqrt_dt is sqrt(dt / 2.) in the predictor and sqrt(dt) in the
 * corrector of a step, sqrt(dt) in advance_qg.  *dts is a float like the reference's. */
static int stochastic_stage(msqg_model *m, double sqrt_dt, float *dts) {
  m->corrector_step = (m->corrector_step + 1) % 2;
  *dts = sqrt_dt;
  if (m->corrector_step) {
    int rc = generate_noise(m);
    if (rc) return rc;
    *dts = *dts / sqrt(2);
  }
  return MSQG_OK;
}

/* advance_qg(output, input, updates = DQ, dt), qg.h:594-606 / qg_stochastic.h:128-149 */
extern "C" int msqg_advance(msqg_model *m, int out_id, int in_id, double dt) {
  CK(cudaSetDevice(m->device));
  List *O = list_by_id(m, out_id), *I = list_by_id(m, in_id);
  if (!O || !I || O->nf != m->nl || I->nf != m->nl) FAIL(MSQG_ERR_ARG, "bad list");
  const Geom &g = m->g[m->depth];
  float dts = 0.f;
  const double *noise = nullptr;
  if (m->p.stochastic) {
    int rc = stochastic_stage(m, sqrt(dt), &dts);
    if (rc) return rc;
    noise = m->nstoch.lev[m->depth];
  }
  dim3 b(64, 4);
  k_advance<<<grid2(g.nx, g.ny, b, m->nl), b, 0, m->stream>>>(O->lev[m->depth], I->lev[m->depth], m->dq.lev[m->depth], noise, g, dt, dts);
  m->launches++;
  if (m->p.nptr > 0) { /* advance_qg runs over (nptr+1)*nl scalars, qg.h:597-603, then boundary(output) */
    List &po = out_id == MSQG_QPRED ? m->ptr_pred : m->ptr, &pi = in_id == MSQG_QPRED ? m->ptr_pred : m->ptr;
    k_advance<<<grid2(g.nx, g.ny, b, po.nf), b, 0, m->stream>>>(po.lev[m->depth], pi.lev[m->depth], m->dptr.lev[m->depth], nullptr, g, dt, 0.f);
    dim3 b2(32, 8);
    k_ghosts<<<grid2(g.nx + 2, g.ny + 2, b2, po.nf), b2, 0, m->stream>>>(po.lev[m->depth], po.nf, g, 1.);
    m->launches += 2;
  }
  CK(cudaGetLastError());
  return MSQG_OK;
}

/* One iteration of [BASILISK] run() (predictor-corrector.h), SURVEY.md 3.1:
 *   dt = dtnext(update(evolving, updates, DT));
 *   advance(predictor, evolving, updates, dt/2); update(predictor, updates, dt);
 *   advance(evolving, evolving, updates, dt)
 * with RHS and stage update fused (k_rhs).  dtnext() [BASILISK] rounds dt so
 * that t lands on tnext_event (pass a negative value for "no pending event"). */
extern "C" int msqg_step(msqg_model *m, double t, double tnext_event, double *dt_out, double *tnext_out) {
  CK(cudaSetDevice(m->device));
  if (m->group) return pg_step(m->group, m, t, tnext_event, dt_out, tnext_out);
  const int D = m->depth;
  int rc;
  /* stage 1 */
  if ((rc = invertq_list(m, m->q))) return rc;
  if ((rc = rhs_prepare(m))) return rc;
  CK(cudaStreamSynchronize(m->stream));
  double tnext;
  double dt = dtnext(t, tnext_event, dt_chain(m, m->h_scal + 1, m->umax_pg, m->p.DT), &tnext);
  float dts = 0.f;
  if (m->p.stochastic && (rc = stochastic_stage(m, sqrt(dt / 2.), &dts))) return rc;
  double *dqp = m->keep_dq ? m->dq.lev[D] : nullptr;
  if ((rc = rhs_launch(m, m->q, m->q.lev[D], m->qpred.lev[D], dqp, dt / 2., dts))) return rc;
  if (m->p.nptr > 0 && (rc = ptr_launch(m, m->ptr, m->ptr.lev[D], m->ptr_pred.lev[D], nullptr, dt / 2.))) return rc;
  /* stage 2 */
  if ((rc = invertq_list(m, m->qpred))) return rc;
  if ((rc = rhs_prepare(m))) return rc;
  if (m->p.stochastic && (rc = stochastic_stage(m, sqrt(dt), &dts))) return rc;
  if ((rc = rhs_launch(m, m->qpred, m->q.lev[D], m->q.lev[D], dqp, dt, dts))) return rc;
  if (m->p.nptr > 0 && (rc = ptr_launch(m, m->ptr_pred, m->ptr.lev[D], m->ptr.lev[D], nullptr, dt))) return rc;
  CK(cudaStreamSynchronize(m->stream));
  (void)dt_chain(m, m->h_scal + 1, m->umax_pg, dt); /* update()'s return value is ignored in stage 2; timestep()'s static state is not */
  if (dt_out) *dt_out = dt;
  if (tnext_out) *tnext_out = tnext;
  return MSQG_OK;
}

/* writestdout, qg.c:101-106 */
/* ------------------------------------------------------------------ multi-scale wavelet filter, msqg/qg.h:509-560 */
/* lists + sig_lev (qg.h:1063-1090: restriction(sig_filt), low-pass flags from the finest level down, then 1 - x),
 * computed on the host with the reference's loop and expression order and uploaded level by level */
static int ensure_filter_lists(msqg_model *m) {
  if (m->filter_vars) return MSQG_OK;
  if (m->px * m->py > 1) FAIL(MSQG_ERR_ARG, "the wavelet filter is not available on decomposed grids");
  const int D = m->depth, nl = m->nl;
  int rc;
  if (!m->qof.nf) {
    if ((rc = alloc_list(m, m->qof, nl, -1., D, D))) return rc;
    if (!m->tmp2.nf && (rc = alloc_list(m, m->tmp2, nl, -1., D, D))) return rc; /* shared with advection_de's ENERGY_CONSERV branch */
    if ((rc = alloc_list(m, m->siglev, 1, 1., 0, D))) return rc;
    if ((rc = alloc_list(m, m->wvs, nl, -1., 0, D - 1))) return rc;
    if ((rc = alloc_list(m, m->wvw, nl, -1., 0, D))) return rc;
  }
  std::vector<std::vector<double>> sf(D + 1), sl(D + 1);
  sf[D] = m->h_sigfilt; /* [y][x] */
  for (int l = D - 1; l >= 0; l--) { /* restriction_average: children (0,0),(0,1),(1,0),(1,1), x outer */
    const int n = 1 << l, nf = 2 * n;
    sf[l].resize((size_t)n * n);
    for (int j = 0; j < n; j++)
      for (int i = 0; i < n; i++) {
        const std::vector<double> &a = sf[l + 1];
        double sum = 0.;
        sum += a[(size_t)(2 * j) * nf + 2 * i];
        sum += a[(size_t)(2 * j + 1) * nf + 2 * i];
        sum += a[(size_t)(2 * j) * nf + 2 * i + 1];
        sum += a[(size_t)(2 * j + 1) * nf + 2 * i + 1];
        sf[l][(size_t)j * n + i] = sum / 4;
      }
  }
  for (int l = D; l >= 0; l--) { /* low pass filter */
    const int n = 1 << l;
    const double Dl = m->p.L0 / n;
    sl[l].resize((size_t)n * n);
    for (int j = 0; j < n; j++)
      for (int i = 0; i < n; i++) {
        double ref_flag = 0;
        if (l < D) {
          const std::vector<double> &ch = sl[l + 1];
          const int nf = 2 * n;
          for (int a = 0; a < 2; a++)      /* child.x */
            for (int b = 0; b < 2; b++)    /* child.y */
              ref_flag += ch[(size_t)(2 * j + b) * nf + 2 * i + a];
        }
        const double s = sf[l][(size_t)j * n + i];
        double v;
        if (ref_flag > 0) v = 1;
        else if (s > 2 * Dl) v = 0;
        else if (s <= 2 * Dl && s > Dl) v = 1 - (s - Dl) / Dl;
        else v = 1;
        sl[l][(size_t)j * n + i] = v;
      }
  }
  for (int l = D; l >= 0; l--) { /* high pass filter */
    for (double &v : sl[l]) v = 1 - v;
    const Geom &g = m->g[l];
    std::vector<double> pad(g.plane, 0.);
    for (int j = 0; j < g.ny; j++)
      for (int i = 0; i < g.nx; i++) pad[GIDX(g.pitch, j, i)] = sl[l][(size_t)j * g.nx + i];
    CK(cudaMemcpyAsync(m->siglev.lev[l], pad.data(), g.plane * sizeof(double), cudaMemcpyHostToDevice, m->stream));
    CK(cudaStreamSynchronize(m->stream));
  }
  m->siglev0 = sl[0][0];
  m->filter_vars = 1;
  return MSQG_OK;
}
/* wavelet_filter(qol = Q, pol, qofl = qof_list, dtflt, nbar = 0) */
static int wavelet_filter(msqg_model *m, List &qof_list, double dtflt) {
  const int D = m->depth, nl = m->nl;
  const Geom &g = m->g[D];
  int rc;
  if ((rc = ensure_filter_lists(m))) return rc;
  const size_t bytes = (size_t)nl * g.plane * sizeof(double);
  CK(cudaMemcpyAsync(m->tmp.lev[D], m->q.lev[D], bytes, cudaMemcpyDeviceToDevice, m->stream)); /* tmp[] = qo[] */
  if ((rc = invertq_list(m, m->q))) return rc;
  dim3 b(32, 8);
  /* restriction({po}) */
  for (int l = D - 1; l >= 0; l--) {
    const double *fine = (l + 1 == D) ? m->psi.lev[D] : m->wvs.lev[l + 1];
    k_restrict<<<grid2(m->g[l].nx, m->g[l].ny, b, nl), b, 0, m->stream>>>(fine, m->wvs.lev[l], m->g[l + 1], m->g[l], -1., 0);
    m->launches++;
  }
  /* wavelet(po, w) and w[] *= sig_lev[] on every level */
  for (int l = D - 1; l >= 0; l--) {
    double *fine = (l + 1 == D) ? m->psi.lev[D] : m->wvs.lev[l + 1];
    k_wavelet<false><<<grid2(m->g[l].nx, m->g[l].ny, b, nl), b, 0, m->stream>>>(m->wvs.lev[l], fine, m->wvw.lev[l + 1], m->siglev.lev[l + 1],
                                                                                 m->g[l], m->g[l + 1], 0);
    m->launches++;
  }
  k_wavelet_root<<<1, 32, 0, m->stream>>>(m->wvs.lev[0], m->wvw.lev[0], m->g[0], m->siglev0, nl, 0);
  /* inverse_wavelet(po, w) */
  k_wavelet_root<<<1, 32, 0, m->stream>>>(m->wvs.lev[0], m->wvw.lev[0], m->g[0], m->siglev0, nl, 1);
  m->launches += 2;
  for (int l = 0; l <= D - 1; l++) {
    double *fine = (l + 1 == D) ? m->psi.lev[D] : m->wvs.lev[l + 1];
    k_wavelet<true><<<grid2(m->g[l].nx, m->g[l].ny, b, nl), b, 0, m->stream>>>(m->wvs.lev[l], fine, m->wvw.lev[l + 1], nullptr, m->g[l], m->g[l + 1],
                                                                                l + 1 == D);
    m->launches++;
  }
  CK(cudaGetLastError());
  if ((rc = msqg_comp_q(m))) return rc; /* comp_q(pol, qol) */
  dim3 b2(64, 4);
  k_filter_mean<<<grid2(g.nx, g.ny, b2, nl), b2, 0, m->stream>>>(qof_list.lev[D], m->tmp.lev[D], m->q.lev[D], g, dtflt, 0);
  m->launches++;
  if (dtflt < 0.0) /* for energy diag: restore qo to prefiltered value (list_copy_deep(tmpl, qol, nl)) */
    CK(cudaMemcpyAsync(m->q.lev[D], m->tmp.lev[D], bytes, cudaMemcpyDeviceToDevice, m->stream));
  CK(cudaGetLastError());
  return MSQG_OK;
}
extern "C" int msqg_wavelet_filter(msqg_model *m, double dtflt) {
  CK(cudaSetDevice(m->device));
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "set_const must be called before the filter");
  int rc = ensure_filter_lists(m);
  if (rc) return rc;
  return wavelet_filter(m, m->qof, dtflt);
}
extern "C" int msqg_invert_filter_mean(msqg_model *m) {
  CK(cudaSetDevice(m->device));
  int rc = ensure_filter_lists(m);
  if (rc) return rc;
  /* invertq(tmpl, qofl): tmpl is the unknown (and the initial guess) */
  const int D = m->depth;
  std::swap(m->psi.lev[D], m->tmp.lev[D]);
  rc = invertq_list(m, m->qof);
  std::swap(m->psi.lev[D], m->tmp.lev[D]);
  return rc;
}
static int ensure_energy_lists(msqg_model *m);
extern "C" int msqg_filter_de_pm(msqg_model *m, double dtflt, double ediag, int pm_field) {
  CK(cudaSetDevice(m->device));
  if (pm_field != MSQG_PO_MFT && pm_field != MSQG_PSI) FAIL(MSQG_ERR_ARG, "filter_de: the mean slot is MSQG_PO_MFT or MSQG_PSI");
  int rc;
  if ((rc = ensure_energy_lists(m))) return rc;
  if ((rc = ensure_filter_lists(m))) return rc;
  if ((rc = wavelet_filter(m, m->tmp2, -dtflt))) return rc;
  const int D = m->depth;
  const Geom &g = m->g[D];
  dim3 b(64, 4);
  k_filter_de<<<grid2(g.nx, g.ny, b, m->nl), b, 0, m->stream>>>(m->de_ft.lev[D], m->tmp2.lev[D],
                                                                (pm_field == MSQG_PSI ? m->psi : m->po_mft).lev[D], g, dtflt, ediag);
  m->launches++;
  CK(cudaGetLastError());
  m->nme_ft = 0;
  return MSQG_OK;
}
extern "C" int msqg_filter_de(msqg_model *m, double dtflt, double ediag) { return msqg_filter_de_pm(m, dtflt, ediag, MSQG_PO_MFT); }

/* ------------------------------------------------------------------ energy diagnostics, msqg/qg_energy.h */
static int ensure_energy_lists(msqg_model *m) { /* set_vars_energy, qg_energy.h:244-253 */
  if (m->energy_vars) return MSQG_OK;
  List *L[7] = {&m->de_bf, &m->de_vd, &m->de_j1, &m->de_j2, &m->de_j3, &m->de_ft, &m->po_mft};
  for (int k = 0; k < 7; k++) {
    int rc = alloc_list(m, *L[k], m->nl, -1., m->depth, m->depth);
    if (rc) return rc;
  }
  m->nme_ft = 0;
  m->energy_vars = 1;
  return MSQG_OK;
}
extern "C" int msqg_reset_energy(msqg_model *m) {
  CK(cudaSetDevice(m->device));
  int rc = ensure_energy_lists(m);
  if (rc) return rc;
  const int ids[6] = {MSQG_DE_BF, MSQG_DE_VD, MSQG_DE_J1, MSQG_DE_J2, MSQG_DE_J3, MSQG_DE_FT};
  for (int k = 0; k < 6; k++) if ((rc = msqg_reset_field(m, ids[k]))) return rc;
  return MSQG_OK;
}
extern "C" int msqg_energy_tend(msqg_model *m, double dt, double ediag) {
  CK(cudaSetDevice(m->device));
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "set_const must be called before energy_tend");
  if (m->g[m->depth].bc) FAIL(MSQG_ERR_ARG, "energy diagnostics are not available on decomposed grids");
  int rc = ensure_energy_lists(m);
  if (rc) return rc;
  const int D = m->depth, nl = m->nl;
  const Geom &g = m->g[D];
  /* comp_del2(pol, zetal, 0., 1.) (:230); dissip_de's comp_del2(zetal, tmpl, 0., 1.) (:159) */
  launch_lap(m->stream, nl, m->psi.lev[D], m->zeta.lev[D], g, nullptr, m->sbcc);
  m->launches++;
  if (m->iRe != 0. || m->iRe4 != 0.) {
    launch_lap(m->stream, nl, m->zeta.lev[D], m->tmp.lev[D], g, nullptr, m->sbcc);
    m->launches++;
  }
  EnergyArgs A;
  memset(&A, 0, sizeof(A));
  A.psi = m->psi.lev[D]; A.zeta = m->zeta.lev[D]; A.tmp = m->tmp.lev[D]; A.pp = m->psipg.lev[D];
  A.zp = m->zetap.lev[D]; A.s = m->str.lev[D];
  A.de_bf = m->de_bf.lev[D]; A.de_vd = m->de_vd.lev[D]; A.de_j1 = m->de_j1.lev[D]; A.de_j2 = m->de_j2.lev[D];
  A.de_j3 = m->de_j3.lev[D]; A.po_mft = m->po_mft.lev[D];
  A.g = g;
  for (int l = 0; l < nl; l++) { A.idh0[l] = m->idh0[l]; A.idh1[l] = m->idh1[l]; }
  A.beta = m->p.beta; A.iRe = m->iRe; A.iRe4 = m->iRe4;
  A.ceks = m->Eks / (m->p.Rom * 2 * m->dhf[0]);
  A.cekb = m->Ekb / (m->p.Rom * 2 * m->dhf[nl - 1]);
  A.dt = dt; A.ediag = ediag;
  A.has_pg = m->has_pg; A.has_zp = m->has_zp; A.nme_ft = m->nme_ft;
  if (m->econs) { /* advection_de's ENERGY_CONSERV branch: comp_q(pol, tmp2l), qg_energy.h:33-35 */
    if (!m->tmp2.nf && (rc = alloc_list(m, m->tmp2, nl, -1., D, D))) return rc;
    dim3 bq(64, 4);
    LayerMetrics M = metrics_of(m);
    NL_SWITCH(nl, k_comp_q<NL><<<grid2(g.nx, g.ny, bq), bq, 0, m->stream>>>(m->psi.lev[D], m->str.lev[D], m->tmp2.lev[D], g, M));
    m->launches++;
    A.qt = m->tmp2.lev[D];
  }
  dim3 b(32, 4);
  NL_SWITCH(nl, k_energy<NL><<<grid2(g.nx, g.ny, b), b, 0, m->stream>>>(A));
  m->launches++;
  CK(cudaGetLastError());
  m->nme_ft += 1;
  return MSQG_OK;
}

extern "C" int msqg_ke1(msqg_model *m, double *ke) {
  CK(cudaSetDevice(m->device));
  const Geom &g = m->g[m->depth];
  dim3 b(16, 16);
  dim3 gr = grid2(g.nx, g.ny, b);
  k_ke_partial<<<gr, b, 0, m->stream>>>(m->psi.lev[m->depth], g, m->d_kepart);
  m->launches++;
  CK(cudaGetLastError());
  std::vector<double> part((size_t)gr.x * gr.y);
  CK(cudaMemcpyAsync(part.data(), m->d_kepart, part.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  double s = 0.;
  for (double v : part) s -= v;
  *ke = s;
  return MSQG_OK;
}

/* tendency of pystep_bfn (qg_bfn.h:46-63, vartype == 1): like update_qg without
 * qforcing; the caller has set q and the signed dissipation coefficients. */
extern "C" int msqg_tendency_bfn(msqg_model *m, double direction) {
  CK(cudaSetDevice(m->device));
  msqg_bfn_direction(m, direction);
  int rc;
  if ((rc = invertq_list(m, m->q))) return rc;
  if ((rc = rhs_prepare(m))) return rc;
  const int hq = m->has_qforc;
  m->has_qforc = 0;
  rc = rhs_launch(m, m->q, nullptr, nullptr, m->dq.lev[m->depth], 0., 0.f);
  m->has_qforc = hq;
  if (rc) return rc;
  CK(cudaStreamSynchronize(m->stream));
  (void)dt_chain(m, m->h_scal + 1, m->umax_pg, m->p.DT); /* advection_pv still runs timestep(): static state advances */
  return MSQG_OK;
}

/* ------------------------------------------------------------------ test hooks */
static int upload_level(msqg_model *m, double *dst, const double *host, int nf, int lev, double sg) {
  const Geom &g = m->g[lev];
  size_t cnt = (size_t)nf * g.nx * g.ny;
  if (cnt > m->stage_doubles) FAIL(MSQG_ERR_ARG, "staging buffer too small");
  CK(cudaMemcpyAsync(m->d_stage, host, cnt * sizeof(double), cudaMemcpyHostToDevice, m->stream));
  dim3 b(32, 8);
  k_pack<<<grid2(g.nx + 2, g.ny + 2, b, nf), b, 0, m->stream>>>(dst, m->d_stage, nf, g, sg);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(m->stream));
  return MSQG_OK;
}
static int download_level(msqg_model *m, double *host, const double *src, int nf, int lev) {
  const Geom &g = m->g[lev];
  size_t cnt = (size_t)nf * g.nx * g.ny;
  dim3 b(32, 8);
  k_unpack<<<grid2(g.nx, g.ny, b, nf), b, 0, m->stream>>>(m->d_stage, src, nf, g);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(host, m->d_stage, cnt * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  return MSQG_OK;
}

/* nsweeps x { relax_layer ; boundary_level } on level `level` with the model's
 * stretching and metrics; a, b host [nl][n][n]. */
extern "C" int msqg_test_relax(msqg_model *m, int level, double *a, const double *b, int nsweeps) {
  CK(cudaSetDevice(m->device));
  if (level < 1 || level > m->depth) FAIL(MSQG_ERR_ARG, "bad level");
  if (!m->const_set || !m->s_uniform) FAIL(MSQG_ERR_ARG, "needs set_const and uniform stretching");
  int rc;
  if ((rc = upload_level(m, m->da.lev[level], a, m->nl, level, -1.))) return rc;
  if ((rc = upload_level(m, m->res.lev[level], b, m->nl, level, -1.))) return rc;
  NL_SWITCH(m->nl, { auto C = relax_coef_layers<NL>(m, level); rc = launch_relax<NL>(m, m->da.lev[level], m->res.lev[level], level, nsweeps, C); });
  if (rc) return rc;
  if ((rc = check_relax_err(m))) return rc;
  return download_level(m, a, m->da.lev[level], m->nl, level);
}
/* scalar Helmholtz relax (modal path) with constant lambda */
extern "C" int msqg_test_relax_scalar(msqg_model *m, int level, double lambda, double *a, const double *b, int nsweeps) {
  CK(cudaSetDevice(m->device));
  if (level < 1 || level > m->depth) FAIL(MSQG_ERR_ARG, "bad level");
  int rc;
  if ((rc = upload_level(m, m->da.lev[level], a, 1, level, -1.))) return rc;
  if ((rc = upload_level(m, m->res.lev[level], b, 1, level, -1.))) return rc;
  auto C = relax_coef_scalar(m, level, lambda);
  if ((rc = launch_relax<1>(m, m->da.lev[level], m->res.lev[level], level, nsweeps, C))) return rc;
  if ((rc = check_relax_err(m))) return rc;
  return download_level(m, a, m->da.lev[level], 1, level);
}
extern "C" int msqg_test_residual(msqg_model *m, const double *a, const double *b, double *res, double *maxres) {
  CK(cudaSetDevice(m->device));
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "needs set_const");
  const int D = m->depth;
  int rc;
  if ((rc = upload_level(m, m->psi.lev[D], a, m->nl, D, -1.))) return rc;
  if ((rc = upload_level(m, m->q.lev[D], b, m->nl, D, -1.))) return rc;
  MgProblem P{m->nl, -1, m->psi.lev[D], m->q.lev[D]};
  if ((rc = mg_residual(m, P, maxres))) return rc;
  return download_level(m, res, m->res.lev[D], m->nl, D);
}
extern "C" int msqg_test_residual_levels(msqg_model *m, int mode, const double *a, const double *b, double *out,
                                         double *maxres, int *bottom) {
  CK(cudaSetDevice(m->device));
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "needs set_const");
  if (mode >= 0 && (!m->p.mode_pv_invert || mode >= m->nl)) FAIL(MSQG_ERR_ARG, "mode %d needs mode_pv_invert and mode < nl", mode);
  const int D = m->depth, nf = mode < 0 ? m->nl : 1;
  int rc;
  if ((rc = upload_level(m, m->psi.lev[D], a, nf, D, -1.))) return rc;
  if ((rc = upload_level(m, m->q.lev[D], b, nf, D, -1.))) return rc;
  MgProblem P{nf, mode, m->psi.lev[D], m->q.lev[D]};
  if ((rc = mg_residual(m, P, maxres))) return rc;
  *bottom = residual_pyr_bottom(m);
  for (int l = D; l >= *bottom; l--) {
    if ((rc = download_level(m, out, m->res.lev[l], nf, l))) return rc;
    out += (size_t)nf * m->g[l].nx * m->g[l].ny;
  }
  return MSQG_OK;
}
extern "C" int msqg_test_restrict(msqg_model *m, int level, const double *fine, double *coarse) {
  CK(cudaSetDevice(m->device));
  if (level < 2 || level > m->depth) FAIL(MSQG_ERR_ARG, "bad level");
  int rc;
  if ((rc = upload_level(m, m->res.lev[level], fine, m->nl, level, -1.))) return rc;
  dim3 b(32, 8);
  k_restrict<<<grid2(m->g[level - 1].nx, m->g[level - 1].ny, b, m->nl), b, 0, m->stream>>>(m->res.lev[level], m->res.lev[level - 1], m->g[level], m->g[level - 1], -1., 0);
  CK(cudaGetLastError());
  return download_level(m, coarse, m->res.lev[level - 1], m->nl, level - 1);
}
extern "C" int msqg_test_prolong(msqg_model *m, int level, const double *coarse, double *fine) {
  CK(cudaSetDevice(m->device));
  if (level < 2 || level > m->depth) FAIL(MSQG_ERR_ARG, "bad level");
  int rc;
  if ((rc = upload_level(m, m->da.lev[level - 1], coarse, m->nl, level - 1, -1.))) return rc;
  dim3 b(32, 8);
  launch_prolong(m->stream, m->nl, m->da.lev[level - 1], m->da.lev[level], m->g[level - 1], m->g[level]);
  CK(cudaGetLastError());
  return download_level(m, fine, m->da.lev[level], m->nl, level);
}

/* arguments of msqg_test_cycles / msqg_group_test_cycles: nrelax in 2..100, the range mg_solve can produce */
static int check_cycle_schedule(int nl, int mode_pv_invert, int mode, const int *nrelax, int ncycles, const double *resa) {
  if (mode < -1 || mode >= nl || (mode >= 0 && !mode_pv_invert)) FAIL(MSQG_ERR_ARG, "mode %d needs mode_pv_invert and mode < nl", mode);
  if (ncycles < 1 || !nrelax || !resa) FAIL(MSQG_ERR_ARG, "a schedule of ncycles >= 1 sweep counts and a resa buffer");
  for (int k = 0; k < ncycles; k++)
    if (nrelax[k] < 2 || nrelax[k] > 100) FAIL(MSQG_ERR_ARG, "nrelax[%d] = %d is outside 2..100", k, nrelax[k]);
  return MSQG_OK;
}
extern "C" int msqg_test_cycles(msqg_model *m, int mode, const int *nrelax, int ncycles, double *resa) {
  CK(cudaSetDevice(m->device));
  int rc = check_cycle_schedule(m->nl, m->p.mode_pv_invert, mode, nrelax, ncycles, resa);
  if (rc) return rc;
  if (m->group) return msqg_group_test_cycles(m->group, mode, nrelax, ncycles, resa);
  if (!m->const_set) FAIL(MSQG_ERR_ARG, "set_const must be called before the cycles");
  const int D = m->depth;
  const size_t pl = m->g[D].plane;
  MgProblem P = mode < 0 ? MgProblem{m->nl, -1, m->psi.lev[D], m->q.lev[D]}
                         : MgProblem{1, mode, m->pm.lev[D] + (size_t)mode * pl, m->qm.lev[D] + (size_t)mode * pl};
  msqg_mgstats st;
  return mg_solve(m, P, 1e-3, &st, nrelax, ncycles, resa);
}

/* exact-division self test: out[i] = div_by(x[i], d[i], 1/d[i]) next to x[i]/d[i] */
__global__ void k_divtest(const double *x, const double *d, double *q_fast, double *q_ieee, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double r = 1. / d[i];
  q_fast[i] = div_by(x[i], d[i], r);
  q_ieee[i] = x[i] / d[i];
}
extern "C" int msqg_test_div(int device, const double *x, const double *d, double *q_fast, double *q_ieee, int n) {
  CK(cudaSetDevice(device));
  double *dx, *dd, *df, *di;
  CK(cudaMalloc(&dx, n * sizeof(double))); CK(cudaMalloc(&dd, n * sizeof(double)));
  CK(cudaMalloc(&df, n * sizeof(double))); CK(cudaMalloc(&di, n * sizeof(double)));
  CK(cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dd, d, n * sizeof(double), cudaMemcpyHostToDevice));
  k_divtest<<<(n + 255) / 256, 256>>>(dx, dd, df, di, n);
  CK(cudaGetLastError());
  CK(cudaMemcpy(q_fast, df, n * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(q_ieee, di, n * sizeof(double), cudaMemcpyDeviceToHost));
  cudaFree(dx); cudaFree(dd); cudaFree(df); cudaFree(di);
  return MSQG_OK;
}

/* One mg_cycle + residual on the model's current (psi, q), timed with CUDA
 * events on the model's stream; reps cycles, average ms.  The iterate keeps
 * converging, which does not change the work per cycle. */
extern "C" int msqg_time_vcycle(msqg_model *m, int nrelax, int reps, double *ms_out) {
  CK(cudaSetDevice(m->device));
  if (!m->const_set || m->p.mode_pv_invert) FAIL(MSQG_ERR_ARG, "needs set_const (layer-coupled mode)");
  if (m->g[m->depth].bc) FAIL(MSQG_ERR_ARG, "msqg_time_vcycle times an undecomposed model");
  const int D = m->depth;
  MgProblem P{m->nl, -1, m->psi.lev[D], m->q.lev[D]};
  double r;
  int rc;
  if ((rc = mg_residual(m, P, &r))) return rc;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  CK(cudaEventRecord(e0, m->stream));
  for (int i = 0; i < reps; i++) {
    if ((rc = mg_cycle(m, P, nrelax))) return rc;
    if ((rc = mg_residual(m, P, &r))) return rc;
  }
  CK(cudaEventRecord(e1, m->stream));
  CK(cudaEventSynchronize(e1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if ((rc = check_relax_err(m))) return rc;
  *ms_out = ms / reps;
  return MSQG_OK;
}

/* per-worker timeline of one relax launch: out[w] = {start ns, end ns, spins, 0} */
extern "C" int msqg_test_relax_profile(msqg_model *m, int level, int nsweeps, long long *out, int max_workers) {
  CK(cudaSetDevice(m->device));
  if (level < 1 || level > m->depth) FAIL(MSQG_ERR_ARG, "bad level");
  if (!m->const_set || !m->s_uniform) FAIL(MSQG_ERR_ARG, "needs set_const and uniform stretching");
  long long *d;
  CK(cudaMalloc(&d, (size_t)max_workers * 12 * sizeof(long long)));
  CK(cudaMemset(d, 0, (size_t)max_workers * 12 * sizeof(long long)));
  m->d_dbg = d;
  int rc;
  NL_SWITCH(m->nl, { auto C = relax_coef_layers<NL>(m, level); rc = launch_relax<NL>(m, m->da.lev[level], m->res.lev[level], level, nsweeps, C); });
  m->d_dbg = nullptr;
  if (rc) return rc;
  if ((rc = check_relax_err(m))) return rc;
  CK(cudaMemcpy(out, d, (size_t)max_workers * 12 * sizeof(long long), cudaMemcpyDeviceToHost));
  cudaFree(d);
  return MSQG_OK;
}

/* per-launch timing: enable, run, then read per-category totals.
 * cats: 0 relax(finest level) 1 relax(coarser levels) 2 residual 3 restrict 4 prolong 5 correct 6 laplacians 7 rhs.
 * aux_sum[0] = total sweeps of the finest-level relax launches. */
extern "C" int msqg_profile_enable(msqg_model *m, int on) {
  CK(cudaSetDevice(m->device));
  CK(cudaStreamSynchronize(m->stream));
  m->prof_on = on; m->prof_recs.clear(); m->prof_next = 0;
  return MSQG_OK;
}
extern "C" int msqg_profile_read(msqg_model *m, double *ms, long *count, long *aux_sum) {
  CK(cudaSetDevice(m->device));
  CK(cudaStreamSynchronize(m->stream));
  for (int c = 0; c < PROF_NCAT; c++) { ms[c] = 0.; count[c] = 0; aux_sum[c] = 0; }
  for (auto &r : m->prof_recs) {
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, r.e0, r.e1));
    ms[r.cat] += t; count[r.cat]++; aux_sum[r.cat] += r.aux;
  }
  m->prof_recs.clear(); m->prof_next = 0;
  return MSQG_OK;
}

/* ------------------------------------------------------------------ ensembles (BASELINE config 5): native driver
 * Members are independent models on one device (replicas only, SURVEY.md 8(e)): own handle, own stream, own noise
 * stream.  One persistent host thread per member issues that member's steps, so the launches and the convergence
 * read-backs of the members interleave on the device; the red-black kernels need no cooperative launch, members
 * overlap freely.  Results are, member by member, the bits of the member run alone. */
struct msqg_ensemble {
  std::vector<msqg_model *> members;
  std::vector<double> t;            /* model time of every member */
  std::vector<double> dt_last;
  std::vector<int> rc;
  std::vector<std::string> err;
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_go, cv_done;
  unsigned long gen = 0;            /* command generation */
  int cmd = 0, arg = 0, done = 0;   /* cmd: 1 step x arg, 2 set_const, 3 quit */
};
static void ensemble_worker(msqg_ensemble *E, int k) {
  unsigned long seen = 0;
  for (;;) {
    int cmd, arg;
    {
      std::unique_lock<std::mutex> lk(E->mu);
      E->cv_go.wait(lk, [&] { return E->gen != seen; });
      seen = E->gen; cmd = E->cmd; arg = E->arg;
    }
    if (cmd == 3) return;
    int rc = MSQG_OK;
    msqg_model *m = E->members[k];
    if (cmd == 2) rc = msqg_set_const(m);
    else
      for (int s = 0; s < arg && rc == MSQG_OK; s++) {
        double dt = 0., tn = 0.;
        rc = msqg_step(m, E->t[k], -1., &dt, &tn);
        if (rc == MSQG_OK) { E->t[k] = tn; E->dt_last[k] = dt; }
      }
    E->rc[k] = rc;
    if (rc) E->err[k] = msqg_last_error(); /* the message lives in this thread */
    {
      std::lock_guard<std::mutex> lk(E->mu);
      E->done++;
    }
    E->cv_done.notify_one();
  }
}
static int ensemble_run(msqg_ensemble *E, int cmd, int arg) {
  const int n = (int)E->members.size();
  {
    std::lock_guard<std::mutex> lk(E->mu);
    E->cmd = cmd; E->arg = arg; E->done = 0; E->gen++;
  }
  E->cv_go.notify_all();
  {
    std::unique_lock<std::mutex> lk(E->mu);
    E->cv_done.wait(lk, [&] { return E->done == n; });
  }
  for (int k = 0; k < n; k++)
    if (E->rc[k]) FAIL(E->rc[k], "member %d: %s", k, E->err[k].c_str());
  return MSQG_OK;
}
extern "C" void msqg_ensemble_destroy(msqg_ensemble *E) {
  if (!E) return;
  if (!E->workers.empty()) {
    {
      std::lock_guard<std::mutex> lk(E->mu);
      E->cmd = 3; E->gen++;
    }
    E->cv_go.notify_all();
    for (std::thread &w : E->workers) w.join();
  }
  for (msqg_model *m : E->members) msqg_destroy(m);
  delete E;
}
/* nmembers models of *p on `device`; seeds[k] (NULL: 1000 + k) seeds member k's noise stream (msqg_seed_noise),
   noise_mode as msqg_set_noise_mode, smoother as msqg_set_smoother */
extern "C" int msqg_ensemble_create(const msqg_params *p, int device, int nmembers, const unsigned *seeds, int noise_mode, int smoother,
                                    msqg_ensemble **out) {
  *out = nullptr;
  if (nmembers < 1 || nmembers > 1024) FAIL(MSQG_ERR_ARG, "an ensemble holds 1..1024 members per device");
  msqg_ensemble *E = new msqg_ensemble();
  for (int k = 0; k < nmembers; k++) {
    msqg_model *m = nullptr;
    int rc = msqg_create(p, device, &m);
    if (!rc) { msqg_seed_noise(m, seeds ? seeds[k] : 1000u + k); rc = p->stochastic ? msqg_set_noise_mode(m, noise_mode) : MSQG_OK; }
    if (!rc) rc = msqg_set_smoother(m, smoother);
    if (rc) { if (m) msqg_destroy(m); msqg_ensemble_destroy(E); return rc; }
    E->members.push_back(m);
  }
  E->t.assign(nmembers, 0.); E->dt_last.assign(nmembers, 0.); E->rc.assign(nmembers, 0); E->err.assign(nmembers, std::string());
  for (int k = 0; k < nmembers; k++) E->workers.emplace_back(ensemble_worker, E, k);
  *out = E;
  return MSQG_OK;
}
extern "C" int msqg_ensemble_size(msqg_ensemble *E) { return (int)E->members.size(); }
extern "C" msqg_model *msqg_ensemble_member(msqg_ensemble *E, int k) {
  return (k >= 0 && k < (int)E->members.size()) ? E->members[k] : nullptr;
}
extern "C" int msqg_ensemble_set_const(msqg_ensemble *E) { return ensemble_run(E, 2, 0); }
/* nsteps predictor-corrector steps of every member, members concurrently; dt_last[k] (may be NULL) = last dt of member k */
extern "C" int msqg_ensemble_step(msqg_ensemble *E, int nsteps, double *dt_last) {
  if (nsteps < 0) FAIL(MSQG_ERR_ARG, "nsteps < 0");
  int rc = ensemble_run(E, 1, nsteps);
  if (dt_last) for (size_t k = 0; k < E->members.size(); k++) dt_last[k] = E->dt_last[k];
  return rc;
}
extern "C" double msqg_ensemble_time(msqg_ensemble *E, int k) { return E->t[k]; }

#include "dist_impl.cuh"
