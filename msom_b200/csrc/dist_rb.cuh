/*
 * dist_rb.cuh -- multigrid cycle of a px x py group of tiles with the red-black smoother (included by model.cu).
 *
 * A red-black half-sweep only reads cells of the other colour, so a decomposed sweep gives the SAME bits as the
 * undecomposed one provided every tile sees current values in its halo -- unlike the reference's lexicographic sweep,
 * whose result depends on the MPI decomposition (msqg/poisson_layer.h:55-65; run as `mpirun -np 16`, msqg/qg.c:12-19).
 * The group therefore reproduces the single-GPU red-black result bit for bit on 1, 2, 4 and 8 GPUs, and it does so with
 * ONE halo exchange per level and cycle instead of one per sweep:
 *
 *   - the planes of a tile carry a frame of MSQG_FRAME cells (layout.cuh); before the nrelax sweeps of a level the
 *     tiles exchange a halo of 2 nrelax + 1 cells of da (and, once per cycle for all levels, 2 nrelax cells of res);
 *     k_relax_rb then runs all sweeps on tile + halo, recomputing the neighbours' border cells: after h half-sweeps the
 *     outermost h halo cells are stale and are simply not used any more (communication-avoiding smoothing);
 *   - one halo cell survives the sweeps, which is what the bilinear prolongation to the next level reads;
 *   - the exchange moves the 4 sides and 4 corners in ONE grouped ncclSend/ncclRecv (8 neighbours) -- corners go
 *     straight to the diagonal neighbour, no x-phase/y-phase;
 *   - levels below the agglomeration threshold (global size < agg_n) are REPLICATED: the restricted residual is
 *     all-gathered (ncclAllGather) and every GPU runs the small coarse solve redundantly, so nothing is scattered back
 *     and no GPU idles while one of them works (SURVEY.md section 5).
 * Scalars: one ncclAllReduce(max) per cycle for the residual norm.
 */
#pragma once

/* ------------------------------------------------------------------ 8-neighbour halo exchange of width w */
struct HaloBox { int x0, x1, y0, y1; };
struct HaloPlan {
  HaloBox send[9], recv[9]; /* index d = (dy + 1) * 3 + (dx + 1); 4 = the tile itself, unused */
  int on[9];                /* neighbour exists */
  long long off[9];         /* offset of this item in the direction's buffer, doubles */
  double *sbuf[9], *rbuf[9];
};
/* ------------------------------------------------------------------ the same exchange through peer memory
 * One process per GPU; every tile's receive area is mapped by its neighbours (CUDA IPC) and the PACK kernel stores the
 * halo straight into the neighbour's memory over NVLink, then raises an arrival flag there; the UNPACK kernel of the
 * neighbour spins on its own flag and scatters the data into the halo frame.  Two launches per exchange (all lists of
 * the exchange in one), no NCCL kernel, no host involvement, replayable inside a CUDA graph:
 *   - the exchange counter lives in device memory (read by pack, advanced by the last block of unpack);
 *   - two receive buffers alternate (parity of the counter): a tile can be at most one exchange ahead of a neighbour,
 *     because its unpack of exchange e waits for the neighbour's pack of e, which follows the neighbour's unpack of e-1;
 *   - flags only grow, spins are bounded (an error word is raised instead of hanging the GPU). */
#define XCHG_MAXITEMS 12 /* da of one level + res of every distributed level (a periodic 8192^2 grid has 8 of them, 9 for nl >= 10) */
#define XCHG_SPIN_NS 4000000000ll
#define XCHG_EPB 1024 /* elements per block: 256 threads x 4 independent loads */
struct XItemDev { double *arr; Geom g; int nf, w, ring; long long off[9]; };
struct XchgArgs {
  XItemDev it[XCHG_MAXITEMS];
  int nitems;
  int on[9];
  int p2p;                /* 1: pack stores into the neighbours' receive areas and raises flags; 0: into local send buffers */
  double *area;           /* my receive area and control words */
  double *dst[9];         /* pack destination by direction: the neighbour's receive area (p2p) or my send buffer */
  double *src[9];         /* unpack source by direction when staged (p2p reads `area`) */
  unsigned long long xcap;
  int seg[XCHG_MAXITEMS * 9 + 1]; /* prefix sums of the block counts of the segments s = item * 9 + direction: a FLAT grid, every
                                     block has work (a (blocks, 9, items) grid sized for the largest side spent 10 us per launch on
                                     scheduling empty blocks for corners and coarse levels) */
  int nblk_dir[9];        /* pack blocks per direction (last-block detection before the flag is raised) */
};
__device__ __forceinline__ unsigned long long *xa_flags(double *area, unsigned long long xcap) { return (unsigned long long *)(area + 2 * 9 * xcap); }
/* words behind the receive space: [0..8] arrival flags, [16] exchange counter, [17] error, [32..40] pack block counters,
   [48] unpack block counter */
__device__ __forceinline__ void halo_box_dev(const Geom &g, int w, int ring, int d, bool recv, int &x0, int &x1, int &y0, int &y1) {
  const int dx = d % 3 - 1, dy = d / 3 - 1;
  const int eL = (ring && !(g.bc & 1)) ? 1 : 0, eR = (ring && !(g.bc & 2)) ? 1 : 0;
  const int eB = (ring && !(g.bc & 4)) ? 1 : 0, eT = (ring && !(g.bc & 8)) ? 1 : 0;
  if (dx < 0) { x0 = recv ? -w : 0; x1 = recv ? 0 : w; }
  else if (dx > 0) { x0 = recv ? g.nx : g.nx - w; x1 = recv ? g.nx + w : g.nx; }
  else { x0 = -eL; x1 = g.nx + eR; }
  if (dy < 0) { y0 = recv ? -w : 0; y1 = recv ? 0 : w; }
  else if (dy > 0) { y0 = recv ? g.ny : g.ny - w; y1 = recv ? g.ny + w : g.ny; }
  else { y0 = -eB; y1 = g.ny + eT; }
}
__device__ __forceinline__ void xchg_segment(const XchgArgs &X, int &it, int &d, int &lb) {
  const int bid = blockIdx.x;
  int sidx = 0;
#pragma unroll 1
  for (int k = 1; k <= X.nitems * 9; k++) sidx += (X.seg[k] <= bid) ? 1 : 0; /* seg is non-decreasing */
  it = sidx / 9; d = sidx % 9; lb = bid - X.seg[sidx];
}
__global__ void __launch_bounds__(256) k_xchg_pack(XchgArgs X) {
  int it, d, lb;
  xchg_segment(X, it, d, lb);
  unsigned long long *w_own = xa_flags(X.area, X.xcap);
  const unsigned long long seqn = *(volatile unsigned long long *)(w_own + 16) + 1;
  const XItemDev &I = X.it[it];
  int x0, x1, y0, y1;
  halo_box_dev(I.g, I.w, I.ring, d, false, x0, x1, y0, y1);
  const int bw = x1 - x0, bh = y1 - y0;
  const long long cnt = (long long)bw * bh, tot = cnt * I.nf;
  /* p2p: the neighbour files what comes from me under ITS direction 8 - d, in the buffer of this exchange's parity */
  double *dst = X.p2p ? X.dst[d] + ((seqn & 1) * 9 + (8 - d)) * X.xcap + I.off[d] : X.dst[d] + I.off[d];
  double v[4];
  long long e[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    e[k] = (long long)lb * XCHG_EPB + k * 256 + threadIdx.x;
    if (e[k] < tot) {
      const int f = (int)(e[k] / cnt);
      const long long r = e[k] - (long long)f * cnt;
      const int y = y0 + (int)(r / bw), x = x0 + (int)(r % bw);
      v[k] = I.arr[(size_t)f * I.g.plane + (long long)(y + 1) * I.g.pitch + MSQG_OX + x];
    }
  }
#pragma unroll
  for (int k = 0; k < 4; k++)
    if (e[k] < tot) dst[e[k]] = v[k];
  if (!X.p2p) return;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int *done = (unsigned int *)(w_own + 32) + d;
    const unsigned int t = atomicAdd(done, 1u);
    if (t == (unsigned int)X.nblk_dir[d] - 1) { /* last block of this direction: everything is on its way, raise the flag */
      *done = 0;
      __threadfence_system();
      unsigned long long *pf = xa_flags(X.dst[d], X.xcap) + (8 - d);
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pf), "l"(seqn) : "memory");
    }
  }
}
__global__ void __launch_bounds__(256) k_xchg_unpack(XchgArgs X) {
  int it, d, lb;
  xchg_segment(X, it, d, lb);
  unsigned long long *w_own = xa_flags(X.area, X.xcap);
  const unsigned long long seqn = *(volatile unsigned long long *)(w_own + 16) + 1;
  if (X.p2p) {
    if (threadIdx.x == 0) {
      unsigned long long v;
      long long t0, t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      for (;;) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(w_own + d) : "memory");
        if (v >= seqn) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > XCHG_SPIN_NS) { *(volatile unsigned long long *)(w_own + 17) = 1ull; break; }
      }
    }
    __syncthreads();
  }
  const XItemDev &I = X.it[it];
  int x0, x1, y0, y1;
  halo_box_dev(I.g, I.w, I.ring, d, true, x0, x1, y0, y1);
  const int bw = x1 - x0, bh = y1 - y0;
  const long long cnt = (long long)bw * bh, tot = cnt * I.nf;
  const double *src = X.p2p ? X.area + ((seqn & 1) * 9 + d) * X.xcap + I.off[d] : X.src[d] + I.off[d];
  double v[4];
  long long e[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    e[k] = (long long)lb * XCHG_EPB + k * 256 + threadIdx.x;
    if (e[k] < tot) v[k] = __ldcv(src + e[k]);
  }
#pragma unroll
  for (int k = 0; k < 4; k++)
    if (e[k] < tot) {
      const int f = (int)(e[k] / cnt);
      const long long r = e[k] - (long long)f * cnt;
      const int y = y0 + (int)(r / bw), x = x0 + (int)(r % bw);
      I.arr[(size_t)f * I.g.plane + (long long)(y + 1) * I.g.pitch + MSQG_OX + x] = v[k];
    }
  if (!X.p2p) return;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int *done = (unsigned int *)(w_own + 48);
    __threadfence();
    const unsigned int t = atomicAdd(done, 1u);
    if (t == gridDim.x - 1) { *done = 0; *(volatile unsigned long long *)(w_own + 16) = seqn; }
  }
}

struct XItem {
  std::vector<double *> arr; /* per local tile */
  std::vector<Geom> geo;
  int nf, w, ring;           /* planes, halo width, 1: straight transfers also carry the ghost ring of physical sides */
};

static void halo_boxes(const Geom &g, int w, int ring, int ix, int iy, int px, int py, HaloPlan &P, int periodic = 0) {
  const int eL = (ring && !(g.bc & 1)) ? 1 : 0, eR = (ring && !(g.bc & 2)) ? 1 : 0;
  const int eB = (ring && !(g.bc & 4)) ? 1 : 0, eT = (ring && !(g.bc & 8)) ? 1 : 0;
  for (int dy = -1; dy <= 1; dy++)
    for (int dx = -1; dx <= 1; dx++) {
      const int d = (dy + 1) * 3 + (dx + 1);
      const int nxx = ix + dx, nyy = iy + dy;
      P.on[d] = !(dx == 0 && dy == 0) && (periodic || (nxx >= 0 && nxx < px && nyy >= 0 && nyy < py));
      HaloBox &s = P.send[d], &r = P.recv[d];
      if (dx < 0) { s.x0 = 0; s.x1 = w; r.x0 = -w; r.x1 = 0; }
      else if (dx > 0) { s.x0 = g.nx - w; s.x1 = g.nx; r.x0 = g.nx; r.x1 = g.nx + w; }
      else { s.x0 = r.x0 = -eL; s.x1 = r.x1 = g.nx + eR; }
      if (dy < 0) { s.y0 = 0; s.y1 = w; r.y0 = -w; r.y1 = 0; }
      else if (dy > 0) { s.y0 = g.ny - w; s.y1 = g.ny; r.y0 = g.ny; r.y1 = g.ny + w; }
      else { s.y0 = r.y0 = -eB; s.y1 = r.y1 = g.ny + eT; }
    }
}

/* all items in one grouped exchange: pack (one launch per item and tile), one send/recv pair per neighbour, unpack */
static int exchange_multi(msqg_group *G, std::vector<XItem> &items) {
  G->exchanges++;
  ProfScope ps_x(G->tiles[0], PROF_XCHG, (int)items.size());
  const int nt = (int)G->tiles.size();
  std::vector<std::vector<HaloPlan>> plans(items.size(), std::vector<HaloPlan>(nt));
  std::vector<std::vector<long long>> tot(nt, std::vector<long long>(9, 0));
  for (size_t it = 0; it < items.size(); it++)
    for (int t = 0; t < nt; t++) {
      msqg_model *m = G->tiles[t];
      HaloPlan &P = plans[it][t];
      if (items[it].w > MSQG_FRAME - 1) FAIL(MSQG_ERR_ARG, "halo width %d exceeds the frame", items[it].w);
      halo_boxes(items[it].geo[t], items[it].w, items[it].ring, m->ix, m->iy, G->px, G->py, P, m->periodic);
      for (int d = 0; d < 9; d++) {
        P.sbuf[d] = m->xsend[d]; P.rbuf[d] = m->xrecv[d];
        P.off[d] = tot[t][d];
        if (P.on[d]) tot[t][d] += (long long)items[it].nf * (P.send[d].x1 - P.send[d].x0) * (P.send[d].y1 - P.send[d].y0);
        if ((size_t)tot[t][d] > m->xcap) FAIL(MSQG_ERR_ARG, "halo exchange buffer too small");
      }
    }
  if (items.size() > XCHG_MAXITEMS) FAIL(MSQG_ERR_ARG, "too many lists in one halo exchange");
  std::vector<XchgArgs> args(nt);
  for (int t = 0; t < nt; t++) {
    msqg_model *m = G->tiles[t];
    XchgArgs &X = args[t];
    memset(&X, 0, sizeof(X));
    X.nitems = (int)items.size(); X.area = m->xarea; X.xcap = m->xcap; X.p2p = G->p2p;
    for (int d = 0; d < 9; d++) {
      X.on[d] = plans[0][t].on[d];
      X.dst[d] = G->p2p ? m->peer_area[d] : m->xsend[d];
      X.src[d] = m->xrecv[d];
      X.nblk_dir[d] = 0;
    }
    int nb = 0;
    for (size_t it = 0; it < items.size(); it++) {
      XItemDev &I = X.it[it];
      I.arr = items[it].arr[t]; I.g = items[it].geo[t]; I.nf = items[it].nf; I.w = items[it].w; I.ring = items[it].ring;
      for (int d = 0; d < 9; d++) {
        I.off[d] = plans[it][t].off[d];
        X.seg[it * 9 + d] = nb;
        if (plans[it][t].on[d]) {
          const long long tot_e = (long long)items[it].nf * (plans[it][t].send[d].x1 - plans[it][t].send[d].x0) * (plans[it][t].send[d].y1 - plans[it][t].send[d].y0);
          const int blocks = (int)((tot_e + XCHG_EPB - 1) / XCHG_EPB);
          nb += blocks; X.nblk_dir[d] += blocks;
        }
      }
    }
    X.seg[items.size() * 9] = nb;
  }
  auto launch = [&](int unpack) { /* every pack before any unpack: local tiles share one stream */
    for (int t = 0; t < nt; t++) {
      const int nb = args[t].seg[items.size() * 9];
      if (nb == 0) continue;
      if (!unpack) k_xchg_pack<<<nb, 256, 0, G->stream>>>(args[t]);
      else k_xchg_unpack<<<nb, 256, 0, G->stream>>>(args[t]);
      G->tiles[t]->launches++;
    }
  };
  launch(0);
  CK(cudaGetLastError());
  if (!G->p2p) {
    if (G->kind == 0) {
      for (int t = 0; t < nt; t++) {
        msqg_model *m = G->tiles[t];
        for (int d = 0; d < 9; d++) {
          if (tot[t][d] == 0) continue;
          const int dx = d % 3 - 1, dy = d / 3 - 1;
          msqg_model *nb = tile_at(G, m->ix + dx, m->iy + dy);
          CK(cudaMemcpyAsync(m->xrecv[d], nb->xsend[8 - d], (size_t)tot[t][d] * sizeof(double), cudaMemcpyDeviceToDevice, G->stream));
        }
      }
    } else {
      msqg_model *m = G->tiles[0];
      /* On a periodic process grid one peer can be the neighbour in several directions (px or py = 2), or the rank
         itself (px or py = 1).  Sends are posted by ascending direction and receives by descending direction: what I
         send towards d arrives at the peer from its direction 8 - d, so the k-th send to a peer meets its k-th receive
         from me.  Directions that wrap onto this rank are device copies. */
      NCK(G->nccl->GroupStart());
      for (int d = 0; d < 9; d++) {
        if (tot[0][d] == 0) continue;
        const int peer = tile_rank(G, m->ix + d % 3 - 1, m->iy + d / 3 - 1);
        if (peer != G->rank) NCK(G->nccl->Send(m->xsend[d], (size_t)tot[0][d], NCCL_DOUBLE, peer, G->comm, G->stream));
      }
      for (int d = 8; d >= 0; d--) {
        if (tot[0][d] == 0) continue;
        const int peer = tile_rank(G, m->ix + d % 3 - 1, m->iy + d / 3 - 1);
        if (peer != G->rank) NCK(G->nccl->Recv(m->xrecv[d], (size_t)tot[0][d], NCCL_DOUBLE, peer, G->comm, G->stream));
      }
      NCK(G->nccl->GroupEnd());
      for (int d = 0; d < 9; d++) {
        if (tot[0][d] == 0) continue;
        const int peer = tile_rank(G, m->ix + d % 3 - 1, m->iy + d / 3 - 1);
        if (peer == G->rank) CK(cudaMemcpyAsync(m->xrecv[d], m->xsend[8 - d], (size_t)tot[0][d] * sizeof(double), cudaMemcpyDeviceToDevice, G->stream));
      }
    }
  }
  launch(1);
  CK(cudaGetLastError());
  return MSQG_OK;
}
static int exchange_one(msqg_group *G, int id, int lev, int w, int ring) {
  std::vector<XItem> items(1);
  XItem &X = items[0];
  for (msqg_model *m : G->tiles) {
    List *L = list_by_id(m, id);
    X.arr.push_back(L->lev[lev]); X.geo.push_back(m->g[lev]); X.nf = L->nf;
  }
  X.w = w; X.ring = ring;
  return exchange_multi(G, items);
}

/* ------------------------------------------------------------------ relax on a tile with deep halos */
/* `sweeps` red-black sweeps on tile + halo: the halo holds h_in valid cells on the internal sides on entry and
 * h_in - 2 sweeps on exit (split into passes of at most NSMAX sweeps; bit-identical to sweeping the whole level) */
template <int NL>
static int relax_rb_tile(msqg_model *m, int lev, int sweeps, int h_in, const RelaxCoef<NL> &C) {
  constexpr int NSMAX = RbCfg<NL>::NSMAX;
  const Geom &g = m->g[lev];
  int left = sweeps, h = h_in;
  while (left > 0) {
    const int passes = (left + NSMAX - 1) / NSMAX;
    const int ns = (left + passes - 1) / passes;
    const int ho = h - 2 * ns;
    if (ho < 0) FAIL(MSQG_ERR_ARG, "halo of %d cells is too thin for %d sweeps", h_in, sweeps);
    const int orange[4] = {(g.bc & 1) ? -ho : 0, g.nx + ((g.bc & 2) ? ho : 0), (g.bc & 4) ? -ho : 0, g.ny + ((g.bc & 8) ? ho : 0)};
    int rc = launch_relax_rb_pass<NL, false>(m, m->da.lev[lev], m->res.lev[lev], lev, ns, C, orange, h);
    if (rc) return rc;
    left -= ns; h = ho;
  }
  return MSQG_OK;
}

__global__ void k_place_all(double *__restrict__ full, Geom gfull, const double *__restrict__ gathered, int hx, int hy, int px,
                            int nranks, int nf) {
  /* gathered = [rank][nf][hy][hx] blocks of level La-1 -> interior of the full padded level */
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  const int rf = blockIdx.z, r = rf / nf, f = rf % nf;
  if (x >= hx || y >= hy) return;
  const int ox = (r % px) * hx, oy = (r / px) * hy;
  full[(size_t)f * gfull.plane + GIDX(gfull.pitch, oy + y, ox + x)] = gathered[(((size_t)r * nf + f) * hy + y) * hx + x];
}

/* a += da on the one-cell halo ring of the INTERNAL sides (cells owned by a neighbouring tile; corners included when both
 * sides are internal); thread t walks the ring: bottom row, top row, left column, right column */
__global__ void k_correct_ring(double *__restrict__ a, const double *__restrict__ da, Geom g) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
  const int nx = g.nx, ny = g.ny;
  int x, y;
  if (t < nx + 2) { x = t - 1; y = -1; }
  else if (t < 2 * (nx + 2)) { x = t - (nx + 2) - 1; y = ny; }
  else if (t < 2 * (nx + 2) + ny) { x = -1; y = t - 2 * (nx + 2); }
  else if (t < 2 * (nx + 2) + 2 * ny) { x = nx; y = t - 2 * (nx + 2) - ny; }
  else return;
  const bool okx = x < 0 ? (g.bc & 1) : (x >= nx ? (g.bc & 2) : true);
  const bool oky = y < 0 ? (g.bc & 4) : (y >= ny ? (g.bc & 8) : true);
  if (!okx || !oky) return; /* beyond a physical side: a ghost, rebuilt by k_ghosts */
  const size_t c = (size_t)f * g.plane + GIDX(g.pitch, y, x);
  a[c] = a[c] + da[c];
}

/* one cycle of the problem P[t] of every tile t: the layer-coupled solve (nl, -1, psi, q) or the scalar Helmholtz
 * solve of one vertical mode (1, mode, plane `mode` of pm, of qm) */
static int g_cycle_rb(msqg_group *G, const std::vector<MgProblem> &P, int nrelax) {
  msqg_model *m0 = G->tiles[0];
  const int D = m0->depth, La = m0->agg_level, nf = P[0].nf, mode = P[0].mode;
  const int nt = (int)G->tiles.size(), nranks = G->px * G->py;
  dim3 b(32, 8);
  int rc;
  /* restriction(res) on the distributed levels, then onto this tile's share of level La-1 */
  for (msqg_model *m : G->tiles) {
    for (int l = D - 1; l >= La; l--) {
      ProfScope ps(m, PROF_RESTRICT, l);
      k_restrict<<<grid2(m->g[l].nx, m->g[l].ny, b, nf), b, 0, G->stream>>>(m->res.lev[l + 1], m->res.lev[l], m->g[l + 1], m->g[l], -1., 0);
      m->launches++;
    }
    k_restrict<<<grid2(m->gpatch.nx, m->gpatch.ny, b, nf), b, 0, G->stream>>>(m->res.lev[La], m->res_patch, m->g[La], m->gpatch, -1., 0);
    k_unpack<<<grid2(m->gpatch.nx, m->gpatch.ny, b, nf), b, 0, G->stream>>>(m->patch_stage, m->res_patch, nf, m->gpatch);
    m->launches += 2;
  }
  CK(cudaGetLastError());
  /* every tile receives every tile's block of level La-1 (all-gather) and assembles the full level */
  const int hx = m0->gpatch.nx, hy = m0->gpatch.ny;
  const size_t blk = (size_t)nf * hx * hy;
  if (G->kind == 0) {
    for (msqg_model *m : G->tiles)
      for (int r = 0; r < nt; r++)
        CK(cudaMemcpyAsync(m->gather_buf + (size_t)r * blk, G->tiles[r]->patch_stage, blk * sizeof(double), cudaMemcpyDeviceToDevice, G->stream));
  } else {
    ProfScope ps_g(m0, PROF_XCHG, 100);
    NCK(G->nccl->AllGather(m0->patch_stage, m0->gather_buf, blk, NCCL_DOUBLE, G->comm, G->stream));
  }
  const int chunk0 = nrelax < 7 ? nrelax : 7;
  /* replicated coarse levels: every tile solves levels 1 .. La-1 (same arithmetic, same bits everywhere) */
  for (msqg_model *m : G->tiles) {
    k_place_all<<<grid2(hx, hy, b, nranks * nf), b, 0, G->stream>>>(m->res.lev[La - 1], m->g[La - 1], m->gather_buf, hx, hy, G->px, nranks, nf);
    m->launches++;
    if ((rc = mg_levels(m, nf, mode, nrelax, La - 1, La - 1))) return rc;
    /* this tile's block of level La-1 plus a one-cell ring (homogeneous dirichlet ghosts evaluated on the fly) */
    k_extract_patch<<<grid2(hx + 2, hy + 2, b, nf), b, 0, G->stream>>>(m->da.lev[La - 1], m->g[La - 1], m->patch_stage, hx, hy, m->ix * hx, m->iy * hy,
                                                                        m->periodic);
    k_load_patch<<<grid2(hx + 2, hy + 2, b, nf), b, 0, G->stream>>>(m->da_patch, m->gpatch, m->patch_stage);
    m->launches += 2;
  }
  CK(cudaGetLastError());
  /* distributed levels: prolongation, ONE halo exchange, all sweeps on tile + halo */
  for (int l = La; l <= D; l++) {
    for (msqg_model *m : G->tiles) {
      ProfScope ps(m, PROF_PROLONG, l);
      if (l == La) launch_prolong(G->stream, nf, m->da_patch, m->da.lev[l], m->gpatch, m->g[l]);
      else launch_prolong(G->stream, nf, m->da.lev[l - 1], m->da.lev[l], m->g[l - 1], m->g[l]);
      m->launches++;
    }
    CK(cudaGetLastError());
    int left = nrelax;
    while (left > 0) {
      const int c = left < 7 ? left : 7;       /* sweeps covered by one exchange: 2c + 1 <= 15 cells of halo */
      const int last = (left - c == 0);
      int w = 2 * c + (last ? 1 : 0);          /* one halo cell must survive the last sweep: the prolongation reads it */
      const Geom &g0 = m0->g[l];
      if (w > g0.nx) w = g0.nx;
      if (w > g0.ny) w = g0.ny;
      if (w < 2 * c) FAIL(MSQG_ERR_ARG, "tiles of level %d are too small for %d fused sweeps (raise agg_n)", l, c);
      std::vector<XItem> items(1);
      for (msqg_model *m : G->tiles) { items[0].arr.push_back(m->da.lev[l]); items[0].geo.push_back(m->g[l]); }
      items[0].nf = nf; items[0].w = w; items[0].ring = 0;
      if (l == La && left == nrelax) {
        /* the halo of res on ALL distributed levels (the sweeps recompute up to 2 nrelax border cells of the neighbours)
           rides in the same exchange: one neighbour synchronisation less per cycle */
        for (int l2 = La; l2 <= D; l2++) {
          XItem X;
          for (msqg_model *m : G->tiles) { X.arr.push_back(m->res.lev[l2]); X.geo.push_back(m->g[l2]); }
          X.nf = nf; X.w = 2 * chunk0; X.ring = 0;
          if (X.w > m0->g[l2].nx) X.w = m0->g[l2].nx;
          if (X.w > m0->g[l2].ny) X.w = m0->g[l2].ny;
          items.push_back(X);
        }
      }
      if ((rc = exchange_multi(G, items))) return rc;
      for (msqg_model *m : G->tiles) {
        ProfScope ps(m, l == D ? PROF_RELAX_FINE : PROF_RELAX_COARSE, c);
        if (mode < 0) {
          NL_SWITCH(m->nl, { auto C = relax_coef_layers<NL>(m, l); rc = relax_rb_tile<NL>(m, l, c, w, C); });
        } else
          rc = relax_rb_tile<1>(m, l, c, w, relax_coef_scalar(m, l, m->lam_lev[(size_t)l * m->nl + mode]));
        if (rc) return rc;
      }
      left -= c;
    }
  }
  /* a += da ; boundary(a) */
  for (int t = 0; t < nt; t++) {
    msqg_model *m = G->tiles[t];
    const Geom &g = m->g[D];
    ProfScope ps(m, PROF_CORRECT, 0);
    k_correct<<<grid2(g.nx, g.ny, b, nf), b, 0, G->stream>>>(P[t].a, m->da.lev[D], g, 1);
    m->launches++;
  }
  CK(cudaGetLastError());
  /* one halo cell of da survived the sweeps: the neighbours' correction of those cells is applied here with the same
     operands (a_halo + da_halo, the bits the owner computes), then the ghosts of the physical sides next to a halo
     column / row are rebuilt from it -- no exchange of psi */
  for (int t = 0; t < nt; t++) {
    msqg_model *m = G->tiles[t];
    const Geom &g = m->g[D];
    k_correct_ring<<<dim3((2 * (g.nx + g.ny + 2) + 255) / 256, nf), 256, 0, G->stream>>>(P[t].a, m->da.lev[D], g);
    k_ghosts<<<grid2(g.nx + 2, g.ny + 2, b, nf), b, 0, G->stream>>>(P[t].a, nf, g, -1.);
    m->launches += 2;
  }
  CK(cudaGetLastError());
  return MSQG_OK;
}
