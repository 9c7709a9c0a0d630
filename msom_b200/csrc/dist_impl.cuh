/*
 * dist_impl.cuh -- 2-D domain decomposition of the msqg timestep (included by model.cu).
 *
 * Every group runs on the same tile machinery: the 8-neighbour halo exchange, the coarse levels and the cycle of
 * dist_rb.cuh.  Only the sweeps of a distributed level depend on the smoother:
 *   lexicographic (smoother 0): the reference built with -D_MPI=1 (msqg/qg.c:12-19).  A relaxation sweep is
 *     lexicographic Gauss-Seidel INSIDE the tile with the neighbours' pre-sweep values in a one-cell halo, refreshed
 *     after every sweep (boundary_level == halo exchange, [BASILISK] C3 of SURVEY.md 2c); every other operator is
 *     order-independent.  This is exactly what oracle/msqg_oracle.c emulates with orc_set_decomp(px, py, agg_n), so
 *     the decomposed GPU path is checked bit for bit against the CPU oracle;
 *   red-black (smoother 1): decomposition independent, deep halos, one exchange per level and cycle (dist_rb.cuh).
 * Levels whose global size is below `agg_n` are gathered onto one tile per process and solved there by the
 * undecomposed multigrid (mg_levels): the arithmetic of the reference's serial solve of those levels.
 *
 * Two back-ends behind the same driver:
 *   local : all tiles live in this process on one device (tests, 1-GPU emulation): direct stores or device copies
 *   nccl  : one tile per process/GPU: direct stores into the neighbours' memory (CUDA IPC) or grouped
 *           ncclSend/ncclRecv on the model stream (NVLink), ncclAllReduce for the 8-byte reductions.  NCCL is loaded
 *           lazily with dlopen.
 */
#pragma once

/* ------------------------------------------------------------------ NCCL, loaded lazily */
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId_t;
struct NcclApi {
  int (*GetUniqueId)(ncclUniqueId_t *);
  int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId_t, int);
  int (*CommDestroy)(ncclComm_t);
  int (*GroupStart)();
  int (*GroupEnd)();
  int (*Send)(const void *, size_t, int, int, ncclComm_t, cudaStream_t);
  int (*Recv)(void *, size_t, int, int, ncclComm_t, cudaStream_t);
  int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t);
  int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t);
  const char *(*GetErrorString)(int);
  bool ok;
};
static NcclApi *nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api.ok ? &api : nullptr;
  tried = true;
  api.ok = false;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return nullptr;
#define NCSYM(f, name) *(void **)(&api.f) = dlsym(h, name); if (!api.f) return nullptr;
  NCSYM(GetUniqueId, "ncclGetUniqueId") NCSYM(CommInitRank, "ncclCommInitRank") NCSYM(CommDestroy, "ncclCommDestroy")
  NCSYM(GroupStart, "ncclGroupStart") NCSYM(GroupEnd, "ncclGroupEnd") NCSYM(Send, "ncclSend") NCSYM(Recv, "ncclRecv")
  NCSYM(AllReduce, "ncclAllReduce") NCSYM(AllGather, "ncclAllGather") NCSYM(GetErrorString, "ncclGetErrorString")
#undef NCSYM
  api.ok = true;
  return &api;
}
#define NCCL_DOUBLE 8 /* ncclFloat64 */
#define NCCL_MAX 2    /* ncclMax */
#define NCK(call)                                                                                   \
  do {                                                                                              \
    int r_ = (call);                                                                                \
    if (r_ != 0) FAIL(MSQG_ERR_CUDA, "%s:%d NCCL: %s", __FILE__, __LINE__, G->nccl->GetErrorString(r_)); \
  } while (0)

extern "C" int msqg_nccl_unique_id(void *out128) {
  NcclApi *a = nccl_api();
  if (!a) FAIL(MSQG_ERR_CUDA, "libnccl.so.2 not found");
  ncclUniqueId_t id;
  int r = a->GetUniqueId(&id);
  if (r) FAIL(MSQG_ERR_CUDA, "ncclGetUniqueId: %s", a->GetErrorString(r));
  memcpy(out128, &id, 128);
  return MSQG_OK;
}

/* ------------------------------------------------------------------ coarse-level patch kernels */
/* scatter: (hx+2) x (hy+2) patch around the tile block of the full level; values outside the
 * domain are the homogeneous-dirichlet ghosts of da (coarse_at with bc = 0) */
__global__ void k_extract_patch(const double *__restrict__ full, Geom gfull, double *__restrict__ dst, int hx, int hy, int ox, int oy,
                                int periodic) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x - 1, y = blockIdx.y * blockDim.y + threadIdx.y - 1, f = blockIdx.z;
  if (x > hx || y > hy) return;
  double v;
  if (periodic) /* sbc = -1: the ring around the block holds the cells across the seam */
    v = full[(size_t)f * gfull.plane + GIDX(gfull.pitch, (oy + y + gfull.ny) % gfull.ny, (ox + x + gfull.nx) % gfull.nx)];
  else
    v = coarse_at(full + (size_t)f * gfull.plane, gfull, ox + x, oy + y);
  dst[((size_t)f * (hy + 2) + y + 1) * (hx + 2) + x + 1] = v;
}
__global__ void k_load_patch(double *__restrict__ dst, Geom gp, const double *__restrict__ src) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x - 1, y = blockIdx.y * blockDim.y + threadIdx.y - 1, f = blockIdx.z;
  if (x > gp.nx || y > gp.ny) return;
  dst[(size_t)f * gp.plane + GIDX(gp.pitch, y, x)] = src[((size_t)f * (gp.ny + 2) + y + 1) * (gp.nx + 2) + x + 1];
}

/* ------------------------------------------------------------------ the group */
struct msqg_group {
  msqg_params p;
  int px, py, agg_n, device, kind; /* kind 0 local, 1 nccl */
  int rb;                          /* red-black smoother (deep halos, dist_rb.cuh); 0: lexicographic */
  int p2p;                         /* halo exchange by direct stores into the neighbours' memory instead of staged copies / NCCL */
  int rank, nranks;
  std::vector<msqg_model *> tiles; /* local: all tiles, index iy*px+ix; nccl: this rank's tile */
  cudaStream_t stream;
  bool own_stream = true;
  NcclApi *nccl;
  ncclComm_t comm;
  double *d_red, *h_red; /* reduction scratch (device / pinned host), 64 doubles */
  double ts_previous;
  msqg_mgstats mgpsi, mgmode[MSQG_MAXL]; /* last solve; per vertical mode (mode_pv_invert) */
  long total_cycles;
  double umax_pg[MSQG_MAXL];
  long exchanges;
  GraphCache graphs;
};

/* periodic groups (sbc = -1): the neighbour across a side of the domain is the tile on the opposite side */
static inline int tile_rank(msqg_group *G, int ix, int iy) { return ((iy + G->py) % G->py) * G->px + (ix + G->px) % G->px; }
static inline msqg_model *tile_at(msqg_group *G, int ix, int iy) {
  return G->kind == 0 ? G->tiles[tile_rank(G, ix, iy)] : G->tiles[0];
}
static int exchange_one(msqg_group *G, int id, int lev, int w, int ring);
static int exchange_list(msqg_group *G, int id, int lev) {
  /* the 8-neighbour exchange, which also carries the ghost ring of the physical sides along the tile edges, so every
     halo cell (corners included) holds exactly the value of the undecomposed field */
  return exchange_one(G, id, lev, 1, 1);
}

/* max over tiles/ranks of n doubles that every tile holds at d_scal + off: enqueue (capturable in a CUDA graph),
 * then finish (synchronises the stream and reads the pinned mirror) */
static int reduce_max_enqueue(msqg_group *G, int off, int n) {
  const int nt = (int)G->tiles.size();
  if (G->kind == 1) {
    msqg_model *m = G->tiles[0];
    ProfScope ps_r(m, PROF_XCHG, 1000);
    NCK(G->nccl->AllReduce(m->d_scal + off, G->d_red, n, NCCL_DOUBLE, NCCL_MAX, G->comm, G->stream));
    CK(to_host(G->stream, G->h_red, G->d_red, n)); /* by a kernel, not a copy engine (see k_to_host) */
    return MSQG_OK;
  }
  for (int t = 0; t < nt; t++)
    CK(to_host(G->stream, G->h_red + (size_t)t * n, G->tiles[t]->d_scal + off, n));
  return MSQG_OK;
}
static int reduce_max_finish(msqg_group *G, int n, double *out) {
  const int nt = (int)G->tiles.size();
  CK(cudaStreamSynchronize(G->stream));
  for (int k = 0; k < n; k++) out[k] = 0.;
  if (G->kind == 1) {
    for (int k = 0; k < n; k++) out[k] = G->h_red[k];
    return MSQG_OK;
  }
  for (int t = 0; t < nt; t++)
    for (int k = 0; k < n; k++) out[k] = fmax(out[k], G->h_red[(size_t)t * n + k]);
  return MSQG_OK;
}
static int reduce_max(msqg_group *G, int off, int n, double *out) {
  int rc = reduce_max_enqueue(G, off, n);
  if (rc) return rc;
  return reduce_max_finish(G, n, out);
}

/* ------------------------------------------------------------------ peer-memory mapping of the neighbours' receive areas */
static int group_setup_p2p(msqg_group *G) {
  const int nt = (int)G->tiles.size();
  if (G->kind == 0) { /* all tiles in this process: plain pointers */
    for (int t = 0; t < nt; t++) {
      msqg_model *m = G->tiles[t];
      for (int d = 0; d < 9; d++) {
        const int dx = d % 3 - 1, dy = d / 3 - 1, ax = m->ix + dx, ay = m->iy + dy;
        m->peer_area[d] = (d != 4 && ax >= 0 && ax < G->px && ay >= 0 && ay < G->py) ? tile_at(G, ax, ay)->xarea : nullptr;
      }
    }
    G->p2p = 1;
    return MSQG_OK;
  }
  /* one process per GPU: all-gather the IPC handles of the receive areas, map the (up to 8) neighbours' */
  msqg_model *m = G->tiles[0];
  cudaIpcMemHandle_t mine;
  if (cudaIpcGetMemHandle(&mine, m->xarea) != cudaSuccess) { cudaGetLastError(); return MSQG_OK; } /* stays on NCCL */
  const size_t hb = sizeof(cudaIpcMemHandle_t);
  char *d_all = nullptr;
  CK(cudaMalloc(&d_all, hb * (G->nranks + 1)));
  CK(cudaMemcpyAsync(d_all + hb * G->nranks, &mine, hb, cudaMemcpyHostToDevice, G->stream));
  NCK(G->nccl->AllGather(d_all + hb * G->nranks, d_all, hb, 0 /* ncclInt8 */, G->comm, G->stream));
  std::vector<cudaIpcMemHandle_t> all(G->nranks);
  CK(cudaMemcpyAsync(all.data(), d_all, hb * G->nranks, cudaMemcpyDeviceToHost, G->stream));
  CK(cudaStreamSynchronize(G->stream));
  cudaFree(d_all);
  int ok = 1;
  for (int d = 0; d < 9 && ok; d++) {
    const int dx = d % 3 - 1, dy = d / 3 - 1, ax = m->ix + dx, ay = m->iy + dy;
    if (d == 4 || ax < 0 || ax >= G->px || ay < 0 || ay >= G->py) continue;
    void *ptr = nullptr;
    if (cudaIpcOpenMemHandle(&ptr, all[tile_rank(G, ax, ay)], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
    m->peer_area[d] = (double *)ptr; m->ipc_opened[d] = ptr;
  }
  /* every rank must take the same path: all-reduce(min) of the outcome */
  double v = ok, *dv = G->d_red;
  CK(cudaMemcpyAsync(dv, &v, sizeof(double), cudaMemcpyHostToDevice, G->stream));
  NCK(G->nccl->AllReduce(dv, dv + 1, 1, NCCL_DOUBLE, 3 /* ncclMin */, G->comm, G->stream));
  CK(cudaMemcpyAsync(&v, dv + 1, sizeof(double), cudaMemcpyDeviceToHost, G->stream));
  CK(cudaStreamSynchronize(G->stream));
  G->p2p = v > 0.5;
  return MSQG_OK;
}
static int group_check_p2p(msqg_group *G) {
  if (!G->p2p) return MSQG_OK;
  for (msqg_model *m : G->tiles) {
    unsigned long long *he = (unsigned long long *)(G->h_red + 64 * 63); /* last row of the pinned scratch */
    CK(to_host(G->stream, he, (const unsigned long long *)(m->xarea + 2 * 9 * m->xcap) + 17, 1));
    CK(cudaStreamSynchronize(G->stream));
    const unsigned long long e = *he;
    if (e) FAIL(MSQG_ERR_CUDA, "peer-memory halo exchange timed out waiting for a neighbour");
  }
  return MSQG_OK;
}

/* ------------------------------------------------------------------ create / destroy */
static int group_create(const msqg_params *p, int device, int px, int py, int agg_n, int kind, int rank, int nranks,
                        const void *uid, msqg_group **out, int smoother = -1) {
  if (smoother < 0) { const char *e = getenv("MSQG_SMOOTHER"); smoother = (e && !strcmp(e, "rb")) ? 1 : 0; }
  *out = nullptr;
  const int per = p->sbc == -1;
  if (px * py < 2 && !per) FAIL(MSQG_ERR_ARG, "a group needs px*py >= 2 tiles");
  if (per && smoother != 1) FAIL(MSQG_ERR_ARG, "periodic boundaries (sbc = -1) need the red-black smoother");
  if (p->mode_pv_invert) {
    /* the vertical-mode inversion runs the red-black cycle once per mode; the lexicographic tile sweep has no modal solve */
    if (smoother != 1) FAIL(MSQG_ERR_ARG, "the vertical-mode inversion (mode_pv_invert) on tiles needs the red-black smoother");
    if (per) FAIL(MSQG_ERR_ARG, "the vertical-mode inversion (mode_pv_invert) is not built for periodic boundaries");
    if (p->varRo > 0)
      FAIL(MSQG_ERR_ARG, "the vertical-mode inversion (mode_pv_invert) on tiles needs uniform vertical modes: varRo > 0 makes them vary with y");
  }
  if (kind == 1 && nranks != px * py) FAIL(MSQG_ERR_ARG, "nranks must equal px*py");
  msqg_group *G = new msqg_group();
  G->p = *p; G->px = px; G->py = py; G->agg_n = agg_n; G->device = device; G->kind = kind;
  G->rank = rank; G->nranks = nranks; G->nccl = nullptr; G->comm = nullptr; G->rb = smoother == 1;
  G->ts_previous = 0.; G->total_cycles = 0; G->exchanges = 0;
  memset(&G->mgpsi, 0, sizeof(G->mgpsi));
  memset(G->mgmode, 0, sizeof(G->mgmode));
  memset(G->umax_pg, 0, sizeof(G->umax_pg));
  CK(cudaSetDevice(device));
  CK(cudaStreamCreateWithFlags(&G->stream, cudaStreamNonBlocking));
  CK(cudaMalloc(&G->d_red, 64 * sizeof(double)));
  CK(cudaHostAlloc(&G->h_red, 64 * 64 * sizeof(double), cudaHostAllocMapped | cudaHostAllocPortable));
  int rc;
  if (kind == 0) {
    for (int iy = 0; iy < py; iy++)
      for (int ix = 0; ix < px; ix++) {
        msqg_model *m;
        /* the levels below agg_n live on tiles[0] only (the solver tile of the process) */
        if ((rc = create_model(p, device, px, py, ix, iy, agg_n, G->stream, &m, G->rb, G->tiles.empty()))) return rc;
        m->smoother = G->rb;
        m->tile_index = (int)G->tiles.size();
        G->tiles.push_back(m);
      }
  } else {
    G->nccl = nccl_api();
    if (!G->nccl) FAIL(MSQG_ERR_CUDA, "libnccl.so.2 not found");
    ncclUniqueId_t id;
    memcpy(&id, uid, 128);
    NCK(G->nccl->CommInitRank(&G->comm, nranks, id, rank));
    msqg_model *m;
    if ((rc = create_model(p, device, px, py, rank % px, rank / px, agg_n, G->stream, &m, G->rb, true))) return rc;
    m->smoother = G->rb;
    G->tiles.push_back(m);
  }
  G->p2p = 0;
  int want = 1;
  { const char *e = getenv("MSQG_P2P"); if (e && atoi(e) == 0) want = 0; }
  if (per) want = 0; /* a tile may be its own neighbour in several directions: staged device copies */
  if (want && (rc = group_setup_p2p(G))) return rc;
  *out = G;
  return MSQG_OK;
}
/* 1: peer-memory halo exchange, 0: staged device copies (local group) or NCCL send/recv */
extern "C" int msqg_group_transport(msqg_group *G) { return G->p2p; }
extern "C" int msqg_group_create_local(const msqg_params *p, int device, int px, int py, int agg_n, msqg_group **out) {
  return group_create(p, device, px, py, agg_n, 0, 0, 1, nullptr, out);
}
extern "C" int msqg_group_create_nccl(const msqg_params *p, int device, int px, int py, int agg_n, int rank, int nranks,
                                      const void *uid128, msqg_group **out) {
  return group_create(p, device, px, py, agg_n, 1, rank, nranks, uid128, out);
}
extern "C" int msqg_group_create_local_sm(const msqg_params *p, int device, int px, int py, int agg_n, int smoother, msqg_group **out) {
  return group_create(p, device, px, py, agg_n, 0, 0, 1, nullptr, out, smoother);
}
extern "C" int msqg_group_create_nccl_sm(const msqg_params *p, int device, int px, int py, int agg_n, int smoother, int rank,
                                         int nranks, const void *uid128, msqg_group **out) {
  return group_create(p, device, px, py, agg_n, 1, rank, nranks, uid128, out, smoother);
}
extern "C" int msqg_group_smoother(msqg_group *G) { return G->rb; }
extern "C" void msqg_group_destroy(msqg_group *G) {
  if (!G) return;
  cudaSetDevice(G->device);
  cudaStreamSynchronize(G->stream);
  G->graphs.clear();
  for (msqg_model *m : G->tiles) msqg_destroy(m);
  if (G->comm && G->nccl) G->nccl->CommDestroy(G->comm);
  cudaFree(G->d_red);
  cudaFreeHost(G->h_red);
  if (G->own_stream) cudaStreamDestroy(G->stream);
  delete G;
}
extern "C" int msqg_group_ntiles(msqg_group *G) { return (int)G->tiles.size(); }
extern "C" msqg_model *msqg_group_tile(msqg_group *G, int t) { return G->tiles[t]; }
extern "C" int msqg_group_tile_info(msqg_group *G, int t, int *info /*ix,iy,x0,y0,nx,ny*/) {
  msqg_model *m = G->tiles[t];
  info[0] = m->ix; info[1] = m->iy; info[2] = m->x0; info[3] = m->y0; info[4] = m->tnx; info[5] = m->tny;
  return MSQG_OK;
}
extern "C" long msqg_group_total_cycles(msqg_group *G) { return G->total_cycles; }
extern "C" long msqg_group_exchanges(msqg_group *G) { return G->exchanges; }
extern "C" long msqg_group_launches(msqg_group *G) { long s = 0; for (msqg_model *m : G->tiles) s += m->launches; return s; }
extern "C" int msqg_group_last_mgstats(msqg_group *G, msqg_mgstats *out) { *out = G->mgpsi; return MSQG_OK; }
extern "C" int msqg_group_last_mode_mgstats(msqg_group *G, int mode, msqg_mgstats *out) {
  if (mode >= G->p.nl) FAIL(MSQG_ERR_ARG, "bad mode");
  *out = mode < 0 ? G->mgpsi : G->mgmode[mode];
  return MSQG_OK;
}
extern "C" int msqg_group_set_stream_sync(msqg_group *G) { CK(cudaStreamSynchronize(G->stream)); return MSQG_OK; }

/* ------------------------------------------------------------------ multigrid on tiles */
/* the problem of every tile: the layer-coupled solve psi <- q_id (mode < 0), or vertical mode `mode`, pm <- qm */
static std::vector<MgProblem> g_problem(msqg_group *G, int mode, int q_id) {
  std::vector<MgProblem> P;
  for (msqg_model *m : G->tiles) {
    const int D = m->depth;
    const size_t pl = m->g[D].plane;
    if (mode < 0) P.push_back(MgProblem{m->nl, -1, m->psi.lev[D], list_by_id(m, q_id)->lev[D]});
    else P.push_back(MgProblem{1, mode, m->pm.lev[D] + (size_t)mode * pl, m->qm.lev[D] + (size_t)mode * pl});
  }
  return P;
}
static int g_residual_enqueue(msqg_group *G, const std::vector<MgProblem> &P) {
  for (int t = 0; t < (int)G->tiles.size(); t++) {
    msqg_model *m = G->tiles[t];
    const int D = m->depth;
    const Geom &g = m->g[D];
    CK(zero_words(G->stream, m->d_scal, 1));
    dim3 b(64, 4);
    ProfScope ps(m, PROF_RESIDUAL, 0);
    if (P[t].mode < 0) {
      LayerMetrics M = metrics_of(m);
      NL_SWITCH(m->nl, k_residual<NL><<<grid2(g.nx, g.ny, b), b, 0, G->stream>>>(P[t].a, P[t].b, m->res.lev[D], m->str.lev[D], g, M, m->d_scal));
    } else
      k_residual_scalar<<<grid2(g.nx, g.ny, b), b, 0, G->stream>>>(P[t].a, P[t].b, m->res.lev[D], m->ibu.lev[D] + (size_t)P[t].mode * g.plane, g,
                                                                   m->d_scal);
    m->launches++;
  }
  CK(cudaGetLastError());
  return reduce_max_enqueue(G, 0, 1);
}
static int g_residual(msqg_group *G, const std::vector<MgProblem> &P, double *maxres) {
  int rc = g_residual_enqueue(G, P);
  if (rc) return rc;
  return reduce_max_finish(G, 1, maxres);
}

static int g_relax_level(msqg_group *G, msqg_model *m, int l, int nsweeps) {
  int rc;
  ProfScope ps(m, l == m->depth ? PROF_RELAX_FINE : PROF_RELAX_COARSE, nsweeps);
  NL_SWITCH(m->nl, { auto C = relax_coef_layers<NL>(m, l); rc = launch_relax<NL>(m, m->da.lev[l], m->res.lev[l], l, nsweeps, C); });
  return rc;
}

static int g_check_err(msqg_group *G) {
  for (msqg_model *m : G->tiles) {
    int rc = check_relax_err(m);
    if (rc) return rc;
  }
  return MSQG_OK;
}

#include "dist_rb.cuh"

/* mg_solve on the decomposed grid: problem P[t] on tile t (NITERMIN 1, NITERMAX 100, nrelax starts at 4); sched as
 * mg_solve's */
static int g_solve(msqg_group *G, const std::vector<MgProblem> &P, msqg_mgstats *st, const int *sched = nullptr,
                   int ncycles = 0, double *resa_out = nullptr) {
  int rc;
  msqg_mgstats s;
  memset(&s, 0, sizeof(s));
  s.nrelax = 4;
  double resb;
  if ((rc = g_residual(G, P, &resb))) return rc;
  s.resb = s.resa = resb;
  for (s.i = 0; sched ? s.i < ncycles : s.i < 100 && (s.i < 1 || s.resa > 1e-3); s.i++) {
    if (sched) s.nrelax = sched[s.i];
    /* one cycle + residual + its all-reduce: with the red-black smoother a single graph launch (keyed by nrelax, the
       mode, the unknown and the right-hand side of tile 0 and the current da buffers of every tile) */
    msqg_model *m0 = G->tiles[0];
    unsigned long long mask = 0;
    for (msqg_model *m : G->tiles) mask = mask * 1315423911ull + da_parity_mask(m);
    bool graphed = G->rb && m0->use_graphs != 0;
    for (msqg_model *m : G->tiles) graphed = graphed && !m->prof_on;
    GraphKey key(s.nrelax, P[0].mode, (const void *)P[0].a, (const void *)P[0].b, mask);
    rc = run_graphed(G->stream, G->graphs, key, G->tiles, &G->exchanges, graphed, [&]() -> int {
      int r2 = g_cycle(G, P, s.nrelax);
      if (r2) return r2;
      return g_residual_enqueue(G, P);
    });
    if (rc) return rc;
    if ((rc = reduce_max_finish(G, 1, &s.resa))) return rc;
    if (sched) resa_out[s.i] = s.resa;
    else if (s.resa > 1e-3) {
      if (resb / s.resa < 1.2 && s.nrelax < 100) s.nrelax++;
      else if (resb / s.resa > 10 && s.nrelax > 2) s.nrelax--;
    }
    resb = s.resa;
  }
  if ((rc = g_check_err(G))) return rc;
  if ((rc = group_check_p2p(G))) return rc;
  G->total_cycles += s.i;
  *st = s;
  return MSQG_OK;
}

/* poisson_layer + invertq on the decomposed grid (invertq_list's order) */
static int g_invertq(msqg_group *G, int q_id) {
  for (msqg_model *m : G->tiles) {
    if (!m->const_set) FAIL(MSQG_ERR_ARG, "set_const must be called before invertq");
    if (!m->s_uniform) FAIL(MSQG_ERR_ARG, "horizontally varying stretching is not supported by the relax kernel yet");
  }
  const int D = G->tiles[0]->depth;
  int rc;
  if (!G->p.mode_pv_invert) {
    if ((rc = exchange_list(G, MSQG_PSI, D))) return rc; /* the warm start's ring */
    return g_solve(G, g_problem(G, -1, q_id), &G->mgpsi);
  }
  /* vertical modes (uniform on tiles: group_create and set_const refuse the others, so the matrices are constants) */
  if ((rc = exchange_list(G, MSQG_PM, D))) return rc; /* the warm start's ring, every mode */
  dim3 b(64, 4), bg(32, 8);
  for (msqg_model *m : G->tiles) {
    const Geom &g = m->g[D];
    NL_SWITCH(m->nl, {
      ModeMat<NL> M;
      for (int k = 0; k < NL * NL; k++) M.a[k] = m->h_cl2m[k];
      k_project<NL><<<grid2(g.nx, g.ny, b), b, 0, G->stream>>>(list_by_id(m, q_id)->lev[D], m->qm.lev[D], g, M, nullptr, 0);
    });
    m->launches++;
  }
  CK(cudaGetLastError());
  for (int l = 0; l < G->p.nl; l++) {
    if ((rc = g_solve(G, g_problem(G, l, q_id), &G->mgmode[l]))) return rc;
    G->mgpsi = G->mgmode[l];
  }
  /* psi on the interior and on the ring of the internal sides: each mode's k_correct_ring left the owner's bits of pm
     there, so the neighbour's psi needs no exchange; then the ghosts of the physical sides */
  for (msqg_model *m : G->tiles) {
    const Geom &g = m->g[D];
    NL_SWITCH(m->nl, {
      ModeMat<NL> M;
      for (int k = 0; k < NL * NL; k++) M.a[k] = m->h_cm2l[k];
      k_project<NL, true><<<grid2(g.nx + 2, g.ny + 2, b), b, 0, G->stream>>>(m->pm.lev[D], m->psi.lev[D], g, M, nullptr, 0);
    });
    k_ghosts<<<grid2(g.nx + 2, g.ny + 2, bg, m->nl), bg, 0, G->stream>>>(m->psi.lev[D], m->nl, g, -1.);
    m->launches += 2;
  }
  CK(cudaGetLastError());
  return MSQG_OK;
}
extern "C" int msqg_group_invertq(msqg_group *G, int q_id) {
  CK(cudaSetDevice(G->device));
  return g_invertq(G, q_id);
}
extern "C" int msqg_group_test_cycles(msqg_group *G, int mode, const int *nrelax, int ncycles, double *resa) {
  CK(cudaSetDevice(G->device));
  int rc = check_cycle_schedule(G->p.nl, G->p.mode_pv_invert, mode, nrelax, ncycles, resa);
  if (rc) return rc;
  for (msqg_model *m : G->tiles) {
    if (!m->const_set) FAIL(MSQG_ERR_ARG, "set_const must be called before the cycles");
    if (mode < 0 && !m->s_uniform) FAIL(MSQG_ERR_ARG, "horizontally varying stretching is not supported by the relax kernel yet");
  }
  if ((rc = exchange_list(G, mode < 0 ? MSQG_PSI : MSQG_PM, G->tiles[0]->depth))) return rc; /* the start's ring, as g_invertq */
  msqg_mgstats st;
  return g_solve(G, g_problem(G, mode, MSQG_Q), &st, nrelax, ncycles, resa);
}

/* ------------------------------------------------------------------ fields, set_const */
extern "C" int msqg_group_set_field(msqg_group *G, int t, int id, const double *host_tile) {
  return msqg_set_field(G->tiles[t], id, host_tile);
}
extern "C" int msqg_group_get_field(msqg_group *G, int t, int id, double *host_tile) {
  return msqg_get_field(G->tiles[t], id, host_tile);
}
/* Uniform vertical modes are computed by every tile from its own Fr (set_const_local): a Fr field that is constant on
 * each tile but differs between tiles would give the tiles different matrices and a wrong result without any error.
 * So every tile and rank must have used the same Fr bits.  reduce_max takes maxima of non-negative words, so each value
 * goes in as its two 32-bit halves h and their complements 2^32 - 1 - h: max(h) + max(2^32 - 1 - h) = 2^32 - 1 exactly
 * when h is the same everywhere. */
static int g_check_modes_agree(msqg_group *G) {
  const int nl = G->p.nl, n = 4 * (nl - 1), nt = (int)G->tiles.size();
  const double ones = 4294967295.;
  std::vector<double> w((size_t)nt * n), out(n);
  for (int t = 0; t < nt; t++) {
    msqg_model *m = G->tiles[t];
    const size_t tc = (size_t)m->tnx * m->tny;
    double *wt = &w[(size_t)t * n];
    for (int l = 0; l < nl - 1; l++) {
      unsigned long long u;
      memcpy(&u, &m->h_fr[(size_t)l * tc], sizeof(u));
      const double hi = (double)(u >> 32), lo = (double)(u & 0xffffffffull);
      wt[4 * l] = hi; wt[4 * l + 1] = ones - hi; wt[4 * l + 2] = lo; wt[4 * l + 3] = ones - lo;
    }
    CK(cudaMemcpyAsync(m->d_scal + 1, wt, n * sizeof(double), cudaMemcpyHostToDevice, G->stream));
  }
  int rc = reduce_max(G, 1, n, out.data());
  if (rc) return rc;
  for (int k = 0; k < n; k += 2)
    if (out[k] + out[k + 1] != ones)
      FAIL(MSQG_ERR_ARG, "Fr of interface %d differs between tiles: the vertical-mode inversion on tiles needs the same Fr "
                         "everywhere (uniform vertical modes)", k / 4);
  return MSQG_OK;
}
extern "C" int msqg_group_set_const(msqg_group *G) {
  CK(cudaSetDevice(G->device));
  G->graphs.clear();
  int rc;
  const int D = G->tiles[0]->depth;
  for (msqg_model *m : G->tiles)
    if ((rc = set_const_local(m))) return rc;
  if (G->p.mode_pv_invert && (rc = g_check_modes_agree(G))) return rc;
  for (int id : {MSQG_PSI, MSQG_PSIPG, MSQG_TOPO})
    if ((rc = exchange_list(G, id, D))) return rc;
  for (msqg_model *m : G->tiles)
    if ((rc = set_const_finish(m))) return rc;
  if ((rc = exchange_list(G, MSQG_ZETAP, D))) return rc;
  /* CFL speeds of the static background flow: max over tiles */
  int has_pg = 0;
  for (msqg_model *m : G->tiles) has_pg |= m->has_pg;
  for (int l = 0; l < G->p.nl; l++) G->umax_pg[l] = 0.;
  if (G->kind == 0) {
    for (msqg_model *m : G->tiles)
      for (int l = 0; l < G->p.nl; l++) G->umax_pg[l] = fmax(G->umax_pg[l], m->umax_pg[l]);
  } else {
    msqg_model *m = G->tiles[0];
    CK(cudaMemcpyAsync(m->d_scal + 1, m->umax_pg, G->p.nl * sizeof(double), cudaMemcpyHostToDevice, G->stream));
    if ((rc = reduce_max(G, 1, G->p.nl, G->umax_pg))) return rc;
  }
  (void)has_pg;
  CK(cudaStreamSynchronize(G->stream));
  return MSQG_OK;
}

/* ------------------------------------------------------------------ RHS and the step */
static int g_rhs_prepare(msqg_group *G, double *umax) {
  const int D = G->tiles[0]->depth;
  int rc;
  dim3 b(64, 4);
  bool use_tmp = false;
  for (msqg_model *m : G->tiles) {
    const Geom &g = m->g[D];
    CK(zero_words(G->stream, m->d_scal + 1, m->nl));
    ProfScope ps(m, PROF_LAP, 0);
    launch_lap(G->stream, m->nl, m->psi.lev[D], m->zeta.lev[D], g, m->d_scal + 1, 0.);
    m->launches++;
    use_tmp = (m->iRe != 0. || m->iRe4 != 0.);
  }
  CK(cudaGetLastError());
  if ((rc = exchange_list(G, MSQG_ZETA, D))) return rc;
  if (use_tmp) {
    for (msqg_model *m : G->tiles) {
      const Geom &g = m->g[D];
      ProfScope ps(m, PROF_LAP, 0);
      launch_lap(G->stream, m->nl, m->zeta.lev[D], m->tmp.lev[D], g, nullptr, 0.);
      m->launches++;
    }
    CK(cudaGetLastError());
    if ((rc = exchange_list(G, MSQG_TMP, D))) return rc;
  }
  return reduce_max(G, 1, G->p.nl, umax);
}
static double g_dt_chain(msqg_group *G, const double *umax, double dtmax) {
  msqg_model *m = G->tiles[0];
  const double Delta = m->g[m->depth].Delta;
  m->ts_previous = G->ts_previous;
  for (int l = 0; l < m->nl; l++) {
    dtmax = timestep_chain(m, umax[l], dtmax, Delta);
    dtmax = timestep_chain(m, G->umax_pg[l], dtmax, Delta);
  }
  G->ts_previous = m->ts_previous;
  return dtmax;
}
/* Stochastic forcing: every tile keeps its own corrector flag, noise mode, seed and draw counter (msqg_seed_noise and
 * msqg_set_noise_mode act on one tile) and all of them advance identically, so the tiles draw, each for its window,
 * the field of the undecomposed model.  Tiles seeded differently would give wrong bits without any error, so at the
 * first stochastic step after a tile's seed or mode changed the group compares mode, seed and draw count across all
 * tiles and ranks, with the complement trick of g_check_modes_agree.  Under NCCL every rank seeds its tile with the
 * same arguments, so every rank takes this check at the same step. */
static int g_check_noise_agree(msqg_group *G) {
  bool pending = false;
  for (msqg_model *m : G->tiles) pending |= !m->noise_agreed;
  if (!pending) return MSQG_OK;
  const int n = 8, nt = (int)G->tiles.size();
  const double ones = 4294967295.;
  std::vector<double> w((size_t)nt * n), out(n);
  for (int t = 0; t < nt; t++) {
    msqg_model *m = G->tiles[t];
    const double h[4] = {(double)m->noise_mode, (double)m->noise_seed, (double)(m->noise_draw >> 32),
                         (double)(m->noise_draw & 0xffffffffull)};
    double *wt = &w[(size_t)t * n];
    for (int k = 0; k < 4; k++) { wt[2 * k] = h[k]; wt[2 * k + 1] = ones - h[k]; }
    CK(cudaMemcpyAsync(m->d_scal + 1, wt, n * sizeof(double), cudaMemcpyHostToDevice, G->stream));
  }
  int rc = reduce_max(G, 1, n, out.data());
  if (rc) return rc;
  static const char *what[4] = {"noise mode", "noise seed", "noise draw count", "noise draw count"};
  for (int k = 0; k < n; k += 2)
    if (out[k] + out[k + 1] != ones)
      FAIL(MSQG_ERR_ARG, "the %s differs between tiles: seed every tile of a stochastic group alike (msqg_seed_noise, "
                         "msqg_set_noise_mode on every tile and rank, with the same arguments)", what[k / 2]);
  for (msqg_model *m : G->tiles) m->noise_agreed = 1;
  return MSQG_OK;
}

extern "C" int msqg_group_step(msqg_group *G, double t, double tnext_event, double *dt_out, double *tnext_out) {
  CK(cudaSetDevice(G->device));
  int rc;
  if (G->p.stochastic && (rc = g_check_noise_agree(G))) return rc;
  double umax[MSQG_MAXL];
  if ((rc = g_invertq(G, MSQG_Q))) return rc;
  if ((rc = g_rhs_prepare(G, umax))) return rc;
  double dt = g_dt_chain(G, umax, G->p.DT);
  double tnext;
  if (tnext_event >= 0 && tnext_event > t) {
    unsigned int nn = (tnext_event - t) / dt;
    tnext = tnext_event;
    if (nn == 0) dt = tnext_event - t;
    else {
      const double dt1 = (tnext_event - t) / nn;
      if (dt1 > dt * (1. + 1e-9)) dt = (tnext_event - t) / (nn + 1);
      else if (dt1 < dt) dt = dt1;
      tnext = t + dt;
    }
  } else
    tnext = t + dt;
  for (msqg_model *m : G->tiles) { /* msqg_step: the noise of each stage is drawn before its right-hand side */
    const int D = m->depth;
    float dts = 0.f;
    if (G->p.stochastic && (rc = stochastic_stage(m, sqrt(dt / 2.), &dts))) return rc;
    if ((rc = rhs_launch(m, m->q, m->q.lev[D], m->qpred.lev[D], nullptr, dt / 2., dts))) return rc;
  }
  if ((rc = g_invertq(G, MSQG_QPRED))) return rc;
  if ((rc = g_rhs_prepare(G, umax))) return rc;
  for (msqg_model *m : G->tiles) {
    const int D = m->depth;
    float dts = 0.f;
    if (G->p.stochastic && (rc = stochastic_stage(m, sqrt(dt), &dts))) return rc;
    if ((rc = rhs_launch(m, m->qpred, m->q.lev[D], m->q.lev[D], nullptr, dt, dts))) return rc;
  }
  CK(cudaStreamSynchronize(G->stream));
  (void)g_dt_chain(G, umax, dt);
  if (dt_out) *dt_out = dt;
  if (tnext_out) *tnext_out = tnext;
  return MSQG_OK;
}
/* CUDA-event timing on the group's stream: which = 0 records the start, 1 records the stop,
 * waits for it and returns the elapsed milliseconds */
extern "C" int msqg_group_timer(msqg_group *G, int which, double *ms) {
  static thread_local cudaEvent_t e0 = nullptr, e1 = nullptr;
  CK(cudaSetDevice(G->device));
  if (!e0) { CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); }
  if (which == 0) { CK(cudaEventRecord(e0, G->stream)); return MSQG_OK; }
  CK(cudaEventRecord(e1, G->stream));
  CK(cudaEventSynchronize(e1));
  float t = 0.f;
  CK(cudaEventElapsedTime(&t, e0, e1));
  if (ms) *ms = t;
  return MSQG_OK;
}
extern "C" int msqg_group_profile_enable(msqg_group *G, int on) {
  for (msqg_model *m : G->tiles) { int rc = msqg_profile_enable(m, on); if (rc) return rc; }
  return MSQG_OK;
}
extern "C" int msqg_group_profile_read(msqg_group *G, double *ms, long *count, long *aux_sum) {
  for (int c = 0; c < PROF_NCAT; c++) { ms[c] = 0.; count[c] = 0; aux_sum[c] = 0; }
  for (msqg_model *m : G->tiles) {
    double a[PROF_NCAT]; long b[PROF_NCAT], c2[PROF_NCAT];
    int rc = msqg_profile_read(m, a, b, c2);
    if (rc) return rc;
    for (int c = 0; c < PROF_NCAT; c++) { ms[c] += a[c]; count[c] += b[c]; aux_sum[c] += c2[c]; }
  }
  return MSQG_OK;
}

/* ------------------------------------------------------------------ a periodic model behind the single-model entry points
 * msqg_create(p with sbc = -1): a local 1 x 1 red-black group whose only tile is the handle the caller gets. */
static int pg_create(const msqg_params *p, int device, msqg_model **out) {
  *out = nullptr;
  msqg_group *G = nullptr;
  int rc = group_create(p, device, 1, 1, 0, 0, 0, 1, nullptr, &G, 1);
  if (rc) { if (G) msqg_group_destroy(G); return rc; }
  msqg_model *m = G->tiles[0];
  m->group = G;
  *out = m;
  return MSQG_OK;
}
static void pg_destroy(msqg_group *G) { msqg_group_destroy(G); }
static int pg_set_stream(msqg_group *G, cudaStream_t s) {
  CK(cudaStreamSynchronize(G->stream));
  G->graphs.clear();
  if (G->own_stream) cudaStreamDestroy(G->stream);
  G->stream = s; G->own_stream = false;
  for (msqg_model *m : G->tiles) { m->graphs.clear(); m->stream = s; m->own_stream = false; }
  return MSQG_OK;
}
static void pg_mirror_stats(msqg_group *G, msqg_model *m) { m->mgpsi = G->mgpsi; m->total_cycles = G->total_cycles; }
static int pg_set_const(msqg_group *G) { return msqg_group_set_const(G); }
static int pg_invertq(msqg_group *G, msqg_model *m, int q_id) {
  int rc = g_invertq(G, q_id);
  pg_mirror_stats(G, m);
  return rc;
}
static int pg_halo(msqg_group *G, int id) { return exchange_list(G, id, G->tiles[0]->depth); }
/* update_qg on the periodic tile: msqg_update with the group's inversion, halo exchanges and dt chain */
static int pg_update(msqg_group *G, msqg_model *m, int q_id, double dtmax, double *dtmax_out) {
  int rc;
  double umax[MSQG_MAXL];
  if ((rc = g_invertq(G, q_id))) return rc;
  pg_mirror_stats(G, m);
  if ((rc = g_rhs_prepare(G, umax))) return rc;
  if ((rc = rhs_launch(m, *list_by_id(m, q_id), nullptr, nullptr, m->dq.lev[m->depth], 0., 0.f))) return rc;
  CK(cudaStreamSynchronize(G->stream));
  if (dtmax_out) *dtmax_out = g_dt_chain(G, umax, dtmax);
  return MSQG_OK;
}
static int pg_step(msqg_group *G, msqg_model *m, double t, double tnext_event, double *dt_out, double *tnext_out) {
  int rc = msqg_group_step(G, t, tnext_event, dt_out, tnext_out);
  pg_mirror_stats(G, m);
  return rc;
}
