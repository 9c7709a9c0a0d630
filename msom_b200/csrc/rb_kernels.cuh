/*
 * rb_kernels.cuh -- throughput smoother of the PV inversion: red-black ordering of relax_layer (sm_100a, fp64).
 *
 * The cell update is the reference's (msqg/poisson_layer.h:80-146: assemble the nl x nl tridiagonal system of one
 * column from the four horizontal neighbours, Thomas solve, write back in place; scalar Helmholtz variant
 * [BASILISK] poisson.h relax(), in-tree copy mspg/elliptic.h:294-301), expression by expression (-fmad=false,
 * divisions by the iterate-independent pivots through div_by(), which returns the IEEE quotient).  Only the
 * TRAVERSAL differs: a sweep is two half-sweeps, cells with (x + y) even ("red") first, then (x + y) odd ("black"),
 * each followed by boundary_level.  The reference documents that the result of its own sweep depends on traversal
 * order, OpenMP and MPI (poisson_layer.h:55-65); a red-black half-sweep only reads cells of the other colour, so its
 * result depends on none of them.  oracle/msqg_oracle.c restates this ordering (orc_set_smoother(m, 1)) and the
 * kernel is bit-exact against it.
 *
 * Temporal blocking: all ns <= 4 sweeps (nh = 2 ns half-sweeps) of a level are ONE pass over HBM.
 *   - a CTA owns an output block of TX = 128 - 2 nh columns x `rpc` rows and streams the rows of its 128-column
 *     window (output block + halo of nh cells on every side that has neighbours) through a shared-memory ring;
 *   - thread (k, p) applies half-sweep k to column pair p (columns 2p, 2p+1 of the window; exactly one of the two has
 *     the colour of half-sweep k in a given row); at step t it works on window row t - 1 - 2k, so half-sweep k runs two
 *     rows behind half-sweep k - 1 and all nh half-sweeps of a step are independent of each other: one
 *     __syncthreads() per step;
 *   - cells whose halo is incomplete (window edge) are computed anyway; the garbage moves inward one cell per
 *     half-sweep and reaches exactly the halo after nh of them -- no validity masks, only the output block is stored;
 *   - rows are fetched with cp.async RB_PF steps ahead and stored column-parity-split ([pair of layers][parity][pair]),
 *     so that every shared-memory access of a warp is a contiguous run of 16-byte words (conflict-free);
 *   - of the four neighbours only north and the one outside the pair are loaded: south and the in-pair neighbour are
 *     the values the thread loaded one step earlier (it moves one row up and switches column every step).
 * HBM traffic per pass: read da and res once (plus halo redundancy 128/TX), write da once, whatever ns is.  The pass
 * is OUT of place (da -> da_out): the output block of one CTA is halo of its neighbours, which must read the
 * pre-pass values; the host swaps the two buffers afterwards.
 * Homogeneous dirichlet ghosts of da are evaluated as -(value of the cell itself before its update), which is what
 * boundary_level left in the ghost ring (the ghost of a cell only mirrors that cell, and the cell only changes in its
 * own half-sweep).
 */
#pragma once
#include "mg_kernels.cuh"

#define RB_WX 128     /* window columns */
#define RB_NP 64      /* column pairs of the window = threads per half-sweep stage */
#define RB_PF 4       /* rows fetched ahead */
#define RB_NSMAX 4    /* sweeps fused in one pass */

struct RbArgs {
  const double *da;   /* in: [NL] planes of the level */
  double *da_out;     /* out: a DIFFERENT buffer of the same geometry (the output block of a CTA is halo of its neighbours) */
  const double *res;  /* rhs of the correction equation */
  Geom g;
  int ns;             /* sweeps of this pass, 1..RB_NSMAX */
  int R;              /* ring rows = 4 ns + 1 + RB_PF */
  int TX;             /* output columns per strip = window columns - 4 ns */
  int rpc;            /* output rows per chunk */
  int ox_lo, ox_hi, oy_lo, oy_hi; /* cells stored by this launch (own cells; a tile may add a ring of halo cells) */
  int xlo, xhi, ylo, yhi;         /* cells that exist in memory: own cells + deep halo on internal sides */
  int par0;           /* parity of the tile origin (x0 + y0) & 1 */
  const double *coef; /* RCOEF: per-row [rows][6][NL] or per-cell [rows][coef_cell][6][NL] Thomas coefficients (k_rowcoef),
                         pointing at the entry of cell (0, 0); a tile's table also holds its halo */
  int coef_cell;      /* RCOEF: entries per row of a per-cell table, 0 = per-row table */
  int reuse;          /* 1: south / in-pair neighbours from registers (default); 0: always from shared memory */
  double *a;          /* k_relax_rb<..., FOLD = true>, last pass on the finest level of an undecomposed grid: the store is
                         a += da with the dirichlet ghost ring of a (k_correct) instead of da_out = da; da_out is not
                         written */
};

__device__ __forceinline__ void cp_async8(unsigned smem_addr, const void *gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(smem_addr), "l"(gsrc));
}

/* sweeps per pass: bounded by the ring (4 ns + 1 + RB_PF rows <= 227 KB) and by registers (threads = 128 ns) */
__host__ __device__ constexpr int rb_nsmax(int nl) { return nl <= 4 ? RB_NSMAX : (nl <= 8 ? 2 : 1); }
/* layer counts with a FOLD instance of k_relax_rb: the single-stage instances (nl > 8) are at the register limit
   already (the prefetched values of a would spill), their finest levels keep the separate k_correct launch */
__host__ __device__ constexpr bool rb_can_fold(int nl) { return rb_nsmax(nl) > 1; }

template <int NL>
struct RbCfg {
  static constexpr int NL2 = (NL + 1) / 2;          /* layer pairs (16-byte words per cell) */
  static constexpr int ARR2 = NL2 * RB_WX;          /* double2 per array per ring row */
  static constexpr int ROW2 = 2 * ARR2;             /* double2 per ring row: da, then res */
  static constexpr size_t row_bytes = (size_t)ROW2 * 16;
  static constexpr int NSMAX = rb_nsmax(NL);
  static_assert((size_t)(4 * NSMAX + 1 + RB_PF) * row_bytes <= 227 * 1024, "ring does not fit");
};

template <int NL, bool RCOEF, bool FOLD = false>
__global__ void __launch_bounds__(RbCfg<NL>::NSMAX * RB_WX, 1)
k_relax_rb(RbArgs A, RelaxCoef<NL> C) {
  using Cfg = RbCfg<NL>;
  constexpr int WX = RB_WX, NP = RB_NP, PF = RB_PF, NSMAX = Cfg::NSMAX;
  constexpr int NL2 = Cfg::NL2, ARR2 = Cfg::ARR2, ROW2 = Cfg::ROW2;
  constexpr int EPT = (2 * NL + NSMAX - 1) / NSMAX; /* planes (da: 0..NL-1, res: NL..2NL-1) streamed per thread */
  constexpr int EPO = (NL + NSMAX - 1) / NSMAX;     /* planes stored per thread */
  static_assert(!FOLD || rb_can_fold(NL), "no FOLD instance for this layer count");
  extern __shared__ double2 ring[];
  /* the block always has NSMAX * 128 threads: stages k >= nh only help with the streaming */
  const int tid = threadIdx.x;
  const int nh = 2 * A.ns, H = nh;
  const int k = tid / NP, p = tid % NP;
  const int pitch = A.g.pitch, nx = A.g.nx, ny = A.g.ny, bc = A.g.bc;
  const long long plane = (long long)A.g.plane;
  /* output block and window of this CTA */
  const int ox0 = A.ox_lo + blockIdx.x * A.TX;
  const int ox1 = min(ox0 + A.TX, A.ox_hi);
  const int x0w = ox0 - H;
  const int oy0 = A.oy_lo + blockIdx.y * A.rpc;
  const int oy1 = min(oy0 + A.rpc, A.oy_hi);
  const int jw0 = max(A.ylo, oy0 - H), jw1 = min(A.yhi, oy1 + H);
  const int nrw = jw1 - jw0; /* window rows */

  /* ---- streaming state: thread <-> window column wx, planes q0 + i * NSMAX; pointers move one row per step */
  const int wx = tid % WX, q0 = tid / WX;
  const int gxl = x0w + wx;
  const bool lvalid = gxl >= A.xlo && gxl < A.xhi;
  const bool ovalid = gxl >= ox0 && gxl < ox1;
  const int colofs = ((wx & 1) * NP + (wx >> 1)) * 2; /* doubles; parity-split column inside a layer-pair block */
  double *ring_d = reinterpret_cast<double *>(ring);
  const unsigned ring_s = (unsigned)__cvta_generic_to_shared(ring_d);
  const double *src[EPT];
  unsigned dofs[EPT];
  bool pok[EPT];
#pragma unroll
  for (int i = 0; i < EPT; i++) {
    const int q = q0 + i * NSMAX;
    pok[i] = lvalid && q < 2 * NL;
    const int arr = q >= NL ? 1 : 0, l = arr ? q - NL : q;
    src[i] = (arr ? A.res : A.da) + (pok[i] ? (long long)l * plane + (long long)(jw0 + 1) * pitch + MSQG_OX + gxl : 0);
    dofs[i] = (unsigned)((arr * 2 * ARR2 + (l >> 1) * 2 * WX + (l & 1) + colofs) * 8);
  }
  const bool corr = FOLD && A.a != nullptr; /* correction out: the store goes to a (+= da), not to da_out */
  double *dst[EPO];
  unsigned sofs[EPO];
  bool sok[EPO];
#pragma unroll
  for (int i = 0; i < EPO; i++) {
    const int q = q0 + i * NSMAX;
    sok[i] = ovalid && q < NL;
    dst[i] = (corr ? A.a : A.da_out) + (sok[i] ? (long long)q * plane + (long long)(jw0 + 1) * pitch + MSQG_OX + gxl : 0);
    sofs[i] = (unsigned)((q >> 1) * 2 * WX + (q & 1) + colofs);
  }
  int ld_row = 0;      /* next window row to fetch */
  unsigned ld_off = 0; /* its ring slot, bytes */
  const unsigned ROWB = (unsigned)Cfg::row_bytes, RTOTB = (unsigned)A.R * ROWB;
  auto load_row = [&]() {
    if (ld_row < nrw) {
#pragma unroll
      for (int i = 0; i < EPT; i++)
        if (pok[i]) { cp_async8(ring_s + ld_off + dofs[i], src[i]); src[i] += pitch; }
    }
    cp_async_commit();
    ld_row++;
    ld_off = ld_off + ROWB == RTOTB ? 0u : ld_off + ROWB;
  };
#pragma unroll 1
  for (int r = 0; r < PF; r++) load_row();

  /* ---- stage state: half-sweep k works on window row r = t - 1 - 2k.  Shared memory is addressed with 32-bit
     byte addresses that move with the row (no generic-pointer arithmetic in the loop). */
  int r = -1 - 2 * k;
  unsigned slB = (unsigned)(((-1 - 2 * k) % A.R + A.R) % A.R) * ROWB; /* ring byte offset of row r */
  int upd = (jw0 + r + k + A.par0 + x0w) & 1;               /* which column of the pair is updated in row r */
  unsigned cuB = (unsigned)(upd * NP + p) * 16u, ciB = (unsigned)((1 - upd) * NP + p) * 16u;
  /* outer neighbour for upd = 0 / 1 (clamped at the window edge: those cells are halo garbage anyway) */
  const unsigned co0B = (unsigned)(NP + (p > 0 ? p - 1 : 0)) * 16u, co1B = (unsigned)(p < NP - 1 ? p + 1 : NP - 1) * 16u;
  const int gxa = x0w + 2 * p, gxb = gxa + 1;
  const bool exa = gxa >= A.xlo && gxa < A.xhi, exb = gxb >= A.xlo && gxb < A.xhi;
  /* physical x-boundaries of this pair: bit 0 = the outer neighbour is a ghost, bit 1 = the in-pair neighbour is */
  const int pl = !(bc & 1), pr = !(bc & 2);
  const int xg0 = ((gxa == 0 && pl) ? 1 : 0) | ((gxa == nx - 1 && pr) ? 2 : 0);  /* upd = 0: west is outer, east in-pair */
  const int xg1 = ((gxb == nx - 1 && pr) ? 1 : 0) | ((gxb == 0 && pl) ? 2 : 0);  /* upd = 1: east is outer, west in-pair */
  const int r_bot = (bc & 4) ? -(1 << 30) : -jw0, r_top = (bc & 8) ? -(1 << 30) : ny - 1 - jw0;
  const bool stage_on = k < nh;
  const bool no_reuse = A.reuse == 0;
  constexpr unsigned LPB = WX * 16u;      /* bytes between layer pairs */
  constexpr unsigned RESB = ARR2 * 16u;   /* byte offset of res inside a ring row */
  /* ---- store state: the row the last half-sweep completed in the previous step */
  int ro = -2 * nh;
  unsigned soB = (unsigned)(((-2 * nh) % A.R + A.R) % A.R) * ROWB;
  const int ro_lo = oy0 - jw0, ro_hi = oy1 - jw0;
  const int T = nrw + 2 * nh;

  /* Of the four neighbours only north and the outer one are loaded: the thread moves one row up and switches column
     every step, so this step's in-pair neighbour is last step's north and this step's south is last step's in-pair
     neighbour: a FIFO of the last three north values, rotated by unrolling three steps (no register moves). */
  double F0[NL], F1[NL], F2[NL];
#pragma unroll
  for (int l = 0; l < NL; l++) { F0[l] = 0.; F1[l] = 0.; F2[l] = 0.; }
  /* correction out: a of the row stored at step t is loaded at step t - 3 (HBM latency under full bandwidth is more
     than one step) into the buffer of step t mod 3, rotated by the same three-step unroll as the FIFO above */
  double A0[EPO], A1[EPO], A2[EPO];
#pragma unroll
  for (int i = 0; i < EPO; i++) { A0[i] = 0.; A1[i] = 0.; A2[i] = 0.; }

  auto step = [&](double (&Fn)[NL], double (&Fi)[NL], double (&Fs)[NL], double (&Av)[EPO]) {
    load_row();
    if (stage_on && (unsigned)r < (unsigned)nrw) {
      const unsigned rowc = ring_s + slB;
      const unsigned rown = ring_s + (slB + ROWB == RTOTB ? 0u : slB + ROWB);
      const unsigned coB = upd ? co1B : co0B;
      double b[NL], vo[NL];
#pragma unroll
      for (int lp = 0; lp < NL2; lp++) {
        const double2 tb = lds2(rowc + RESB + lp * LPB + cuB);
        const double2 tn = lds2(rown + lp * LPB + cuB);
        const double2 to = lds2(rowc + lp * LPB + coB);
        b[2 * lp] = tb.x; Fn[2 * lp] = tn.x; vo[2 * lp] = to.x;
        if (2 * lp + 1 < NL) { b[2 * lp + 1] = tb.y; Fn[2 * lp + 1] = tn.y; vo[2 * lp + 1] = to.y; }
      }
      if (r == 0 || no_reuse) { /* first row of the window: nothing carried yet */
        const unsigned rows = ring_s + (slB == 0 ? RTOTB - ROWB : slB - ROWB);
#pragma unroll
        for (int lp = 0; lp < NL2; lp++) {
          const double2 ti = lds2(rowc + lp * LPB + ciB);
          const double2 ts = lds2(rows + lp * LPB + cuB);
          Fi[2 * lp] = ti.x; Fs[2 * lp] = ts.x;
          if (2 * lp + 1 < NL) { Fi[2 * lp + 1] = ti.y; Fs[2 * lp + 1] = ts.y; }
        }
      }
      /* relax_layer, poisson_layer.h:80-146 (same expression order as k_relax_ws):
         rhs = -sq(Delta)*b; rhs += a[1] + a[-1]; rhs += a[0,1] + a[0,-1] */
      double sh[NL], sv[NL];
      const int xg = upd ? xg1 : xg0;
      const bool gb = r == r_bot, gt = r == r_top;
      if (xg != 0 || gb || gt) {
        /* homogeneous dirichlet ghosts on the physical sides: -(this cell before its update) */
#pragma unroll
        for (int lp = 0; lp < NL2; lp++) {
          const double2 tc = lds2(rowc + lp * LPB + cuB);
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const int l = 2 * lp + h;
            if (l < NL) {
              const double g = h ? -tc.y : -tc.x;
              const double o = (xg & 1) ? g : vo[l], i = (xg & 2) ? g : Fi[l];
              const double s_ = gb ? g : Fs[l], n_ = gt ? g : Fn[l];
              sh[l] = i + o;
              sv[l] = n_ + s_;
            }
          }
        }
      } else {
#pragma unroll
        for (int l = 0; l < NL; l++) { sh[l] = Fi[l] + vo[l]; sv[l] = Fn[l] + Fs[l]; }
      }
      double rhs[NL], out[NL];
#pragma unroll
      for (int l = 0; l < NL; l++) {
        double rr = C.msd2 * b[l];
        rr += sh[l];
        rr += sv[l];
        rhs[l] = rr;
      }
      if (!RCOEF) {
#pragma unroll
        for (int l = 1; l < NL; l++) rhs[l] -= div_by(C.t0[l] * rhs[l - 1], C.t1p[l - 1], C.rinv[l - 1]);
        out[NL - 1] = div_by(rhs[NL - 1], C.t1p[NL - 1], C.rinv[NL - 1]);
#pragma unroll
        for (int l = NL - 2; l >= 0; l--) out[l] = div_by(rhs[l] - C.t2[l] * out[l + 1], C.t1p[l], C.rinv[l]);
      } else {
        /* horizontally varying stretching: coefficients of this row / cell from the k_rowcoef table, which covers the
           cells that exist (a tile's table also covers its halo); window cells beyond them are garbage anyway */
        const int j = jw0 + r, gx = upd ? gxb : gxa;
        const int jc = min(max(j, A.ylo), A.yhi - 1), xc = min(max(gx, A.xlo), A.xhi - 1);
        const double *ct = A.coef + (A.coef_cell ? (long long)jc * A.coef_cell + xc : (long long)jc) * 6 * NL;
        double t0[NL], t2[NL], t1p[NL], rinv[NL];
#pragma unroll
        for (int l = 0; l < NL; l++) { t0[l] = ct[l]; t2[l] = ct[NL + l]; t1p[l] = ct[2 * NL + l]; rinv[l] = ct[3 * NL + l]; }
#pragma unroll
        for (int l = 1; l < NL; l++) rhs[l] -= div_by(t0[l] * rhs[l - 1], t1p[l - 1], rinv[l - 1]);
        out[NL - 1] = div_by(rhs[NL - 1], t1p[NL - 1], rinv[NL - 1]);
#pragma unroll
        for (int l = NL - 2; l >= 0; l--) out[l] = div_by(rhs[l] - t2[l] * out[l + 1], t1p[l], rinv[l]);
      }
      if (upd ? exb : exa) {
#pragma unroll
        for (int lp = 0; lp < NL2; lp++)
          sts2(rowc + lp * LPB + cuB, out[2 * lp], (2 * lp + 1 < NL) ? out[2 * lp + 1] : 0.);
      }
    }
    r++;
    slB = slB + ROWB == RTOTB ? 0u : slB + ROWB;
    upd ^= 1;
    { const unsigned tmp = cuB; cuB = ciB; ciB = tmp; }
    /* ---- store the row completed in the previous step */
    if (ro >= ro_lo && ro < ro_hi) {
#pragma unroll
      for (int i = 0; i < EPO; i++)
        if (sok[i]) {
          double v;
          asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(ring_s + soB + sofs[i] * 8u));
          if (FOLD && corr) {
            /* k_correct: a += da (a first), then the dirichlet ghost ring of a: -w on the sides, +w at the corners */
            const double w = Av[i] + v;
            double *pa = dst[i];
            *pa = w;
            const int gy = jw0 + ro;
            const bool gl = gxl == 0, gr = gxl == nx - 1, gb = gy == 0, gt = gy == ny - 1;
            if (gl) pa[-1] = -w;
            if (gr) pa[1] = -w;
            if (gb) pa[-pitch] = -w;
            if (gt) pa[pitch] = -w;
            if (gl && gb) pa[-pitch - 1] = w;
            if (gl && gt) pa[pitch - 1] = w;
            if (gr && gb) pa[-pitch + 1] = w;
            if (gr && gt) pa[pitch + 1] = w;
          } else {
            *dst[i] = v;
          }
        }
    }
    if (FOLD && corr && ro + 3 >= ro_lo && ro + 3 < ro_hi) { /* a of the row stored three steps later (ro starts <= -4) */
      const int ahead = ro >= 0 ? 3 : ro + 3;                  /* dst points at row max(ro, 0) */
#pragma unroll
      for (int i = 0; i < EPO; i++)
        if (sok[i]) Av[i] = dst[i][(long long)ahead * pitch];
    }
    if (ro >= 0) {
#pragma unroll
      for (int i = 0; i < EPO; i++) dst[i] += pitch;
    }
    ro++;
    soB = soB + ROWB == RTOTB ? 0u : soB + ROWB;
    cp_async_wait<PF - 1>();
    __syncthreads();
  };

#pragma unroll 1
  for (int t = 0; t < T; t += 3) {
    step(F0, F2, F1, A0);
    if (t + 1 < T) step(F1, F0, F2, A1);
    if (t + 2 < T) step(F2, F1, F0, A2);
  }
  cp_async_wait<0>();
}

/* ------------------------------------------------------------------ the coarsest levels in ONE launch
 * Levels 1 .. Lc (2 x 2 .. 32 x 32 cells) hold 0.01 % of the cells of a 4096^2 hierarchy but cost a dozen latency-bound
 * launches per cycle when swept one by one.  One CTA keeps da and res of all of them in shared memory and runs the
 * cycle's coarse end by itself ([BASILISK] mg_cycle, in-tree copy mspg/elliptic.h:43-99, with red-black sweeps):
 *     res[l] = restriction(res[l+1])                 l = Lc-1 .. 1     (restriction_average, same summation order)
 *     da[1] = 0;  da[l] = bilinear(da[l-1])          l = 2 .. Lc       (same expression as k_prolong4)
 *     nrelax x { red half-sweep ; black half-sweep } on every level    (same cell update as k_relax_rb)
 * Input: res on level Lc (global memory); output: da on level Lc.  Bit-identical to the level-by-level kernels. */
#define RB_COARSE_MAXLEV 5
template <int NL>
struct CoarseCoef { RelaxCoef<NL> c[RB_COARSE_MAXLEV + 1]; }; /* index = level */
struct CoarseArgs {
  const double *res; /* level Lc, [NL] planes */
  double *da;        /* level Lc, [NL] planes */
  Geom g;            /* geometry of level Lc (undecomposed) */
  int Lc, nrelax;
  const double *coef[RB_COARSE_MAXLEV + 1]; /* RCOEF: Thomas coefficient table of every level (k_rowcoef / k_modecoef), else unused */
  int coef_cell;     /* RCOEF: 1 = per cell [ny][nx][6][NL], 0 = per row [ny][6][NL] */
  int periodic;      /* sbc = -1: neighbours and bilinear stencils wrap around instead of meeting dirichlet ghosts */
};
template <int NL>
__device__ __forceinline__ size_t coarse_smem_doubles(int Lc) {
  size_t cells = 0;
  for (int l = 1; l <= Lc; l++) cells += (size_t)1 << (2 * l);
  return 2 * (size_t)NL * cells;
}
template <int NL, bool RCOEF = false>
__global__ void __launch_bounds__(512)
k_coarse_rb(CoarseArgs A, CoarseCoef<NL> CC) {
  extern __shared__ double csm[];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int Lc = A.Lc;
  /* level l: da at base[l], res right behind it; planes [NL][n][n] without ghosts */
  int base[RB_COARSE_MAXLEV + 2];
  {
    int o = 0;
    for (int l = 1; l <= Lc; l++) { base[l] = o; o += 2 * NL * (1 << (2 * l)); }
  }
  auto DA = [&](int l, int f, int y, int x) -> double & { const int n = 1 << l; return csm[base[l] + (f * n + y) * n + x]; };
  auto RS = [&](int l, int f, int y, int x) -> double & { const int n = 1 << l; return csm[base[l] + NL * n * n + (f * n + y) * n + x]; };
  { /* res of level Lc from global memory */
    const int n = 1 << Lc;
    for (int e = tid; e < NL * n * n; e += nt) {
      const int f = e / (n * n), y = (e / n) % n, x = e % n;
      RS(Lc, f, y, x) = A.res[(size_t)f * A.g.plane + GIDX(A.g.pitch, y, x)];
    }
  }
  __syncthreads();
  for (int l = Lc - 1; l >= 1; l--) { /* restriction_average: children (0,0), (0,1) [y+1], (1,0) [x+1], (1,1), then /4 */
    const int n = 1 << l;
    for (int e = tid; e < NL * n * n; e += nt) {
      const int f = e / (n * n), y = (e / n) % n, x = e % n;
      double sum = 0.;
      sum += RS(l + 1, f, 2 * y, 2 * x);
      sum += RS(l + 1, f, 2 * y + 1, 2 * x);
      sum += RS(l + 1, f, 2 * y, 2 * x + 1);
      sum += RS(l + 1, f, 2 * y + 1, 2 * x + 1);
      RS(l, f, y, x) = sum / 4;
    }
    __syncthreads();
  }
  for (int l = 1; l <= Lc; l++) {
    const int n = 1 << l;
    if (l == 1) {
      for (int e = tid; e < NL * n * n; e += nt) csm[base[1] + e] = 0.;
    } else { /* bilinear: (9 C + 3 (C[cx,0] + C[0,cy]) + C[cx,cy]) / 16, homogeneous dirichlet ghosts by reflection */
      const int nc = n >> 1;
      for (int e = tid; e < NL * n * n; e += nt) {
        const int f = e / (n * n), y = (e / n) % n, x = e % n;
        const int xc = x >> 1, yc = y >> 1, ix = (x & 1) ? 1 : -1, iy = (y & 1) ? 1 : -1;
        auto cat = [&](int xx, int yy) {
          double s = 1.;
          if (A.periodic) { xx = (xx + nc) & (nc - 1); yy = (yy + nc) & (nc - 1); }
          else {
            if (xx < 0) { xx = 0; s = -s; } else if (xx >= nc) { xx = nc - 1; s = -s; }
            if (yy < 0) { yy = 0; s = -s; } else if (yy >= nc) { yy = nc - 1; s = -s; }
          }
          return s * DA(l - 1, f, yy, xx);
        };
        DA(l, f, y, x) = (9. * cat(xc, yc) + 3. * (cat(xc + ix, yc) + cat(xc, yc + iy)) + cat(xc + ix, yc + iy)) / 16.;
      }
    }
    __syncthreads();
    const RelaxCoef<NL> &C = CC.c[l];
    const int half = n >> 1; /* cells of one colour per row */
    for (int hs = 0; hs < 2 * A.nrelax; hs++) {
      const int colour = hs & 1;
      for (int e = tid; e < n * half; e += nt) {
        const int y = e / half, x = 2 * (e % half) + ((y + colour) & 1);
        double rhs[NL], out[NL];
#pragma unroll
        for (int f = 0; f < NL; f++) {
          const double c0 = DA(l, f, y, x), gh = -c0;
          double aw, ae, as, an;
          if (A.periodic) { /* the ghost ring holds the opposite side (refreshed after every half-sweep; those cells
                               have the other colour, so they are current) */
            aw = DA(l, f, y, (x + n - 1) & (n - 1)); ae = DA(l, f, y, (x + 1) & (n - 1));
            as = DA(l, f, (y + n - 1) & (n - 1), x); an = DA(l, f, (y + 1) & (n - 1), x);
          } else {
            aw = x > 0 ? DA(l, f, y, x - 1) : gh; ae = x < n - 1 ? DA(l, f, y, x + 1) : gh;
            as = y > 0 ? DA(l, f, y - 1, x) : gh; an = y < n - 1 ? DA(l, f, y + 1, x) : gh;
          }
          double rr = C.msd2 * RS(l, f, y, x);
          rr += ae + aw;
          rr += an + as;
          rhs[f] = rr;
        }
        if (!RCOEF) {
#pragma unroll
          for (int f = 1; f < NL; f++) rhs[f] -= div_by(C.t0[f] * rhs[f - 1], C.t1p[f - 1], C.rinv[f - 1]);
          out[NL - 1] = div_by(rhs[NL - 1], C.t1p[NL - 1], C.rinv[NL - 1]);
#pragma unroll
          for (int f = NL - 2; f >= 0; f--) out[f] = div_by(rhs[f] - C.t2[f] * out[f + 1], C.t1p[f], C.rinv[f]);
        } else { /* horizontally varying stretching / lambda: the coefficients of this row or cell (same tables as k_relax_rb) */
          const double *ct = A.coef[l] + (A.coef_cell ? (size_t)y * n + x : (size_t)y) * 6 * NL;
          double t0[NL], t2[NL], t1p[NL], rinv[NL];
#pragma unroll
          for (int f = 0; f < NL; f++) { t0[f] = ct[f]; t2[f] = ct[NL + f]; t1p[f] = ct[2 * NL + f]; rinv[f] = ct[3 * NL + f]; }
#pragma unroll
          for (int f = 1; f < NL; f++) rhs[f] -= div_by(t0[f] * rhs[f - 1], t1p[f - 1], rinv[f - 1]);
          out[NL - 1] = div_by(rhs[NL - 1], t1p[NL - 1], rinv[NL - 1]);
#pragma unroll
          for (int f = NL - 2; f >= 0; f--) out[f] = div_by(rhs[f] - t2[f] * out[f + 1], t1p[f], rinv[f]);
        }
#pragma unroll
        for (int f = 0; f < NL; f++) DA(l, f, y, x) = out[f];
      }
      __syncthreads();
    }
  }
  { /* da of level Lc to global memory */
    const int n = 1 << Lc;
    for (int e = tid; e < NL * n * n; e += nt) {
      const int f = e / (n * n), y = (e / n) % n, x = e % n;
      A.da[(size_t)f * A.g.plane + GIDX(A.g.pitch, y, x)] = DA(Lc, f, y, x);
    }
  }
}

/* ------------------------------------------------------------------ small levels: one window per CTA, no streaming
 * The streaming kernel pays 2 nh rows of halo and 2 nh steps of pipeline fill per row chunk, which dominates on levels
 * (or tiles) of a few hundred cells per side.  Here a CTA loads the whole window of its RB_TO x RB_TO output block
 * (+ nh cells of halo on every side that has neighbours) into shared memory, runs the nh half-sweeps with one
 * __syncthreads() each -- half-sweep h only touches the cells whose halo is still complete, a region that shrinks by
 * one ring per half-sweep -- and stores the block.  Same cell update, same ghost rule, same bits as k_relax_rb. */
#define RB_TO 32
template <int NL, bool RCOEF = false>
__global__ void __launch_bounds__(512)
k_relax_rb_tile(RbArgs A, RelaxCoef<NL> C) {
  extern __shared__ double tsm[];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int nh = 2 * A.ns, H = nh;
  const int nx = A.g.nx, ny = A.g.ny, bc = A.g.bc, pitch = A.g.pitch;
  const long long plane = (long long)A.g.plane;
  const int ox0 = A.ox_lo + blockIdx.x * RB_TO, ox1 = min(ox0 + RB_TO, A.ox_hi);
  const int oy0 = A.oy_lo + blockIdx.y * RB_TO, oy1 = min(oy0 + RB_TO, A.oy_hi);
  /* window = output block + halo, clipped to the cells that exist */
  const int wx0 = max(A.xlo, ox0 - H), wx1 = min(A.xhi, ox1 + H);
  const int wy0 = max(A.ylo, oy0 - H), wy1 = min(A.yhi, oy1 + H);
  const int ww = wx1 - wx0, wh = wy1 - wy0;
  constexpr int WS = RB_TO + 4 * RB_NSMAX;      /* window pitch */
  double *sda = tsm, *srs = tsm + NL * WS * WS; /* [NL][WS][WS] each */
  for (int e = tid; e < NL * wh * ww; e += nt) {
    const int f = e / (wh * ww), r = e - f * wh * ww, y = r / ww, x = r - y * ww;
    const long long g = (long long)f * plane + (long long)(wy0 + y + 1) * pitch + MSQG_OX + wx0 + x;
    sda[(f * WS + y) * WS + x] = A.da[g];
    srs[(f * WS + y) * WS + x] = A.res[g];
  }
  __syncthreads();
  /* sides of the window that are sides of the whole field: no ring is lost there (ghosts instead of neighbours) */
  const bool eL = wx0 == 0 && !(bc & 1), eR = wx1 == nx && !(bc & 2), eB = wy0 == 0 && !(bc & 4), eT = wy1 == ny && !(bc & 8);
  for (int hs = 0; hs < nh; hs++) {
    const int colour = hs & 1;
    const int lx = eL ? 0 : hs + 1, hx = eR ? ww : ww - hs - 1, ly = eB ? 0 : hs + 1, hy = eT ? wh : wh - hs - 1;
    const int rw = hx - lx, rh = hy - ly, hw = (rw + 1) >> 1;
    for (int e = tid; e < rh * hw; e += nt) {
      const int y = ly + e / hw;
      int x = lx + 2 * (e % hw);
      x += ((wx0 + x + wy0 + y + A.par0) & 1) != colour; /* first cell of this colour at or after x */
      if (x >= hx) continue;
      const int gx = wx0 + x, gy = wy0 + y;
      double rhs[NL], out[NL];
#pragma unroll
      for (int f = 0; f < NL; f++) {
        const double *p = sda + (f * WS + y) * WS + x;
        const double c0 = p[0], gh = -c0;
        const double aw = (gx == 0 && !(bc & 1)) ? gh : (x > 0 ? p[-1] : c0);
        const double ae = (gx == nx - 1 && !(bc & 2)) ? gh : (x < ww - 1 ? p[1] : c0);
        const double as = (gy == 0 && !(bc & 4)) ? gh : (y > 0 ? p[-WS] : c0);
        const double an = (gy == ny - 1 && !(bc & 8)) ? gh : (y < wh - 1 ? p[WS] : c0);
        double rr = C.msd2 * srs[(f * WS + y) * WS + x];
        rr += ae + aw;
        rr += an + as;
        rhs[f] = rr;
      }
      if (!RCOEF) {
#pragma unroll
        for (int f = 1; f < NL; f++) rhs[f] -= div_by(C.t0[f] * rhs[f - 1], C.t1p[f - 1], C.rinv[f - 1]);
        out[NL - 1] = div_by(rhs[NL - 1], C.t1p[NL - 1], C.rinv[NL - 1]);
#pragma unroll
        for (int f = NL - 2; f >= 0; f--) out[f] = div_by(rhs[f] - C.t2[f] * out[f + 1], C.t1p[f], C.rinv[f]);
      } else { /* coefficients of this row / cell from the k_rowcoef / k_modecoef table (it covers every cell of the window) */
        const double *ct = A.coef + (A.coef_cell ? (long long)gy * A.coef_cell + gx : (long long)gy) * 6 * NL;
        double t0[NL], t2[NL], t1p[NL], rinv[NL];
#pragma unroll
        for (int f = 0; f < NL; f++) { t0[f] = ct[f]; t2[f] = ct[NL + f]; t1p[f] = ct[2 * NL + f]; rinv[f] = ct[3 * NL + f]; }
#pragma unroll
        for (int f = 1; f < NL; f++) rhs[f] -= div_by(t0[f] * rhs[f - 1], t1p[f - 1], rinv[f - 1]);
        out[NL - 1] = div_by(rhs[NL - 1], t1p[NL - 1], rinv[NL - 1]);
#pragma unroll
        for (int f = NL - 2; f >= 0; f--) out[f] = div_by(rhs[f] - t2[f] * out[f + 1], t1p[f], rinv[f]);
      }
#pragma unroll
      for (int f = 0; f < NL; f++) sda[(f * WS + y) * WS + x] = out[f];
    }
    __syncthreads();
  }
  const int bw = ox1 - ox0, bh = oy1 - oy0;
  for (int e = tid; e < NL * bh * bw; e += nt) {
    const int f = e / (bh * bw), r = e - f * bh * bw, y = r / bw, x = r - y * bw;
    A.da_out[(long long)f * plane + (long long)(oy0 + y + 1) * pitch + MSQG_OX + ox0 + x] =
        sda[(f * WS + (oy0 + y - wy0)) * WS + (ox0 + x - wx0)];
  }
}
