/*
 * mg_kernels.cuh -- multigrid kernels of the PV inversion (sm_100a, fp64).
 *
 * Replaces, bit for bit in IEEE fp64 (compile with -fmad=false):
 *   residual_layer     msqg/poisson_layer.h:157-258
 *   relax_layer        msqg/poisson_layer.h:48-150   (lexicographic Gauss-Seidel,
 *                      vertical Thomas solve per column, reference sweep order)
 *   [BASILISK] restriction / bilinear / boundary_level / mg_cycle's "a += da"
 *                      (in-tree copy of the cycle: mspg/elliptic.h:43-99)
 *   [BASILISK] poisson.h relax/residual for the modal scalar Helmholtz solves
 *                      (older in-tree copy mspg/elliptic.h:265-359)
 */
#pragma once
#include "layout.cuh"
#include <cuda_runtime.h>
#include <type_traits>

#define FULLMASK 0xffffffffu

/* ------------------------------------------------------------------ small helpers */
__device__ __forceinline__ void atomic_max_pos(double *addr, double v) {
  /* v >= 0 and never NaN: IEEE order == unsigned integer order */
  atomicMax((unsigned long long *)addr, (unsigned long long)__double_as_longlong(v));
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULLMASK, v, o));
  return v;
}

/* Block-wide max of non-negative values -> one atomic per block. */
__device__ __forceinline__ void block_max_to(double *dst, double v) {
  __shared__ double sh[32];
  v = warp_max(v);
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int lane = tid & 31, wid = tid >> 5;
  const int nw = (blockDim.x * blockDim.y + 31) >> 5;
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  if (wid == 0) {
    v = lane < nw ? sh[lane] : 0.;
    v = warp_max(v);
    if (lane == 0 && v > 0.) atomic_max_pos(dst, v);
  }
}

/* Correctly rounded x/d for a divisor whose correctly rounded reciprocal
 * r = RN(1/d) is known.  Two Newton-Markstein corrections: after the first, q is
 * a faithful quotient; the second (exact remainder via FMA) then yields
 * RN(x/d) (Markstein's theorem), i.e. the same bits as the IEEE division the
 * reference performs.  Used on the Thomas-solve critical path where d (the
 * pivot) does not depend on the iterate. */
__device__ __forceinline__ double div_by(double x, double d, double r) {
  double q = x * r;
  double e = __fma_rn(-d, q, x);
  q = __fma_rn(e, r, q);
  e = __fma_rn(-d, q, x);
  q = __fma_rn(e, r, q);
  return q;
}

/* ------------------------------------------------------------------ pack / unpack
 * pyset_field + boundary()  (msqg/qg.h:1164-1175): host-layout [nf][n][n] ->
 * padded planes incl. ghost ring.  sg = -1: dirichlet(0) (msqg/layer.h:17-21),
 * sg = +1: Basilisk default symmetry.  Corner ghosts = sg*sg*corner cell
 * ([BASILISK] box boundaries sweep the full tangential range, x before y). */
__global__ void k_pack(double *__restrict__ dst, const double *__restrict__ src, int nf, Geom g, double sg) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x - 1;
  const int y = blockIdx.y * blockDim.y + threadIdx.y - 1;
  const int f = blockIdx.z;
  if (x > g.nx || y > g.ny) return;
  int xs = x, ys = y;
  double s = 1.;
  if (x < 0) { xs = 0; s *= sg; } else if (x >= g.nx) { xs = g.nx - 1; s *= sg; }
  if (y < 0) { ys = 0; s *= sg; } else if (y >= g.ny) { ys = g.ny - 1; s *= sg; }
  dst[(size_t)f * g.plane + GIDX(g.pitch, y, x)] = s * src[((size_t)f * g.ny + ys) * g.nx + xs];
}

__global__ void k_unpack(double *__restrict__ dst, const double *__restrict__ src, int nf, Geom g) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= g.nx || y >= g.ny) return;
  dst[((size_t)f * g.ny + y) * g.nx + x] = src[(size_t)f * g.plane + GIDX(g.pitch, y, x)];
}

/* boundary_level on a padded list: ghost ring from the interior on the PHYSICAL sides of the tile
 * (sides in g.bc are internal: their ghosts belong to the halo exchange and are left alone).
 * Corner ghosts next to an internal side are filled from that side's ghost column/row, which is how
 * [BASILISK]'s x-then-y boundary sweeps build them; call after the halo exchange. */
__global__ void k_ghosts(double *__restrict__ a, int nf, Geom g, double sg) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x - 1;
  const int y = blockIdx.y * blockDim.y + threadIdx.y - 1;
  const int f = blockIdx.z;
  if (x > g.nx || y > g.ny) return;
  const bool gx = (x < 0 || x >= g.nx), gy = (y < 0 || y >= g.ny);
  if (!gx && !gy) return;
  const bool xin = (x < 0) ? (g.bc & 1) : (x >= g.nx ? (g.bc & 2) : 0);
  const bool yin = (y < 0) ? (g.bc & 4) : (y >= g.ny ? (g.bc & 8) : 0);
  if ((gx && xin && !gy) || (gy && yin && !gx)) return;       /* pure halo cell */
  if (gx && gy && xin && yin) return;                          /* corner owned by the diagonal neighbour */
  int xs = x, ys = y;
  double s = 1.;
  if (gx && !xin) { xs = x < 0 ? 0 : g.nx - 1; s *= sg; }
  if (gy && !yin) { ys = y < 0 ? 0 : g.ny - 1; s *= sg; }
  double *p = a + (size_t)f * g.plane;
  p[GIDX(g.pitch, y, x)] = s * p[GIDX(g.pitch, ys, xs)];
}

/* ------------------------------------------------------------------ residual_layer
 * msqg/poisson_layer.h:182-241 (non-TREE branch, alpha = unity):
 *   res = b -/+ stretching + (fgx(a,0) - fgx(a,1))/Delta + (fgy(a,0) - fgy(a,1))/Delta
 * face_gradient_x(a,i) = (a[i]-a[i-1])/Delta [BASILISK].  max|res| by warp
 * shuffles + one atomic per block.  res ghosts are never read (relax reads the
 * centre, restriction the interior) so they are not written. */
/* dirichlet / symmetry ghosts of a boundary cell (value v, sign sg), corners keep +v (layer.h:17-21 through [BASILISK]) */
__device__ __forceinline__ void write_ghosts_d(double *__restrict__ p, const Geom &g, int x, int y, double v, double sg) {
  const int nx = g.nx, ny = g.ny;
  const bool l = x == 0, r = x == nx - 1, bo = y == 0, t = y == ny - 1;
  if (l) p[GIDX(g.pitch, y, -1)] = sg * v;
  if (r) p[GIDX(g.pitch, y, nx)] = sg * v;
  if (bo) p[GIDX(g.pitch, -1, x)] = sg * v;
  if (t) p[GIDX(g.pitch, ny, x)] = sg * v;
  if (l && bo) p[GIDX(g.pitch, -1, -1)] = v;
  if (l && t) p[GIDX(g.pitch, ny, -1)] = v;
  if (r && bo) p[GIDX(g.pitch, -1, nx)] = v;
  if (r && t) p[GIDX(g.pitch, ny, nx)] = v;
}

struct LayerMetrics {
  double idh0[MSQG_NLMAX], idh1[MSQG_NLMAX];
};

/* The per-cell expressions of the residual, shared by every residual kernel so that the association order is written
 * once.  res_vertical: b and the stretching term of layer l out of NL (NL == 1: b alone); sm / sp = stretching of the
 * interfaces above / below the layer (l - 1, l), am / ap = a of the layers l - 1, l + 1 (ignored where absent). */
template <int NL>
__device__ __forceinline__ double res_vertical(int l, double b, double sm, double sp, double am, double ac, double ap,
                                               const LayerMetrics &M) {
  if (NL == 1) return b;
  if (l == 0) return b + sp * (ac - ap) * M.idh1[0];
  if (l < NL - 1) return b + sm * (ac - am) * M.idh0[l] - sp * (ap - ac) * M.idh1[l];
  return b + sm * (ac - am) * M.idh0[l];
}
/* r + the face-gradient Laplacian of a (x then y); x/Delta via div_by: same bits as the IEEE division, 6x fewer
 * instructions */
__device__ __forceinline__ double res_laplacian(double r, double ac, double aw, double ae, double as, double an, double D,
                                                double rD) {
  r += div_by(div_by(ac - aw, D, rD) - div_by(ae - ac, D, rD), D, rD);
  r += div_by(div_by(ac - as, D, rD) - div_by(an - ac, D, rD), D, rD);
  return r;
}

template <int NL>
__global__ void __launch_bounds__(256)
k_residual(const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ res,
           const double *__restrict__ s, Geom g, LayerMetrics M, double *__restrict__ maxres) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  double m = 0.;
  if (x < g.nx && y < g.ny) {
    const size_t c = GIDX(g.pitch, y, x);
    const double D = g.Delta, rD = g.rD;
    double ac[NL];
#pragma unroll
    for (int l = 0; l < NL; l++) ac[l] = a[l * g.plane + c];
#pragma unroll
    for (int l = 0; l < NL; l++) {
      const double *al = a + l * g.plane;
      const double sm = l > 0 ? s[(l - 1) * g.plane + c] : 0., sp = l < NL - 1 ? s[l * g.plane + c] : 0.;
      double r = res_vertical<NL>(l, b[l * g.plane + c], sm, sp, l > 0 ? ac[l > 0 ? l - 1 : 0] : 0., ac[l],
                                  l < NL - 1 ? ac[l < NL - 1 ? l + 1 : l] : 0., M);
      r = res_laplacian(r, ac[l], al[c - 1], al[c + 1], al[c - g.pitch], al[c + g.pitch], D, rD);
      res[l * g.plane + c] = r;
      const double f = fabs(r);
      if (f > m) m = f;
    }
  }
  block_max_to(maxres, m);
}

/* ------------------------------------------------------------------ residual + restriction pyramid
 * The residual of k_residual (NL >= 2, SFIELD: stretching read from its field, else the per-layer constants S.s of a
 * horizontally uniform field) or of k_residual_scalar (NL == 1: b - lambda a, lambda read from its plane), and from the
 * same tile the restriction of res down the hierarchy (k_restrict's expression, each level from the one above it):
 * levels D-1 .. D-5 of a 32x32 fine tile, as far as P.nlev says.  Undecomposed levels only (g.bc == 0, nx = ny = 2^D).
 *   one thread = one 2x2 quad of fine cells = one cell of level D-1: the first restriction is in registers;
 *   one warp = 16x2 quads: level D-2 by three shuffles, its 8 cells go to shared memory;
 *   one CTA = 8 warps = 32x32 fine cells: levels D-3 (4x4), D-4 (2x2), D-5 (1x1) from shared memory at the end.
 * Rows are read and written as 16-byte pairs (the interior of a row starts 128-byte aligned, a quad at an even x).  The
 * layers are walked in order; a layer needs the centre values of its two neighbours only. */
#define PYR_MAXLEV 5
#define PYR_TILE 32
struct PyrLevels {
  double *p[PYR_MAXLEV]; /* res on levels D-1, D-2, ... */
  int pitch[PYR_MAXLEV];
  size_t plane[PYR_MAXLEV];
  int n[PYR_MAXLEV];     /* cells per side */
  int nlev;              /* levels written below D (0 .. PYR_MAXLEV) */
};
struct StretchConsts {
  double s[MSQG_NLMAX];
};

__device__ __forceinline__ double restrict4(double c00, double c01, double c10, double c11) {
  /* restriction_average, k_restrict's order: (0,0), (0,1) [y+1], (1,0) [x+1], (1,1); the leading 0. maps -0 to +0 */
  double sum = 0.;
  sum += c00;
  sum += c01;
  sum += c10;
  sum += c11;
  return sum / 4;
}

/* one shared-memory stage of the pyramid: W x W cells per layer of the CTA from the (2W) x (2W) of the stage above,
 * kept in dst (unless null) for the next stage and stored on pyramid level k */
template <int NL, int W>
__device__ __forceinline__ void pyr_stage(const double *src, double *dst, const PyrLevels &P, int k, int tid) {
  if (tid < NL * W * W) {
    const int l = tid / (W * W), y = (tid / W) % W, x = tid % W;
    const double *s = src + (l * 2 * W + 2 * y) * 2 * W + 2 * x;
    const double v = restrict4(s[0], s[2 * W], s[1], s[2 * W + 1]);
    if (dst) dst[(l * W + y) * W + x] = v;
    const int gx = blockIdx.x * W + x, gy = blockIdx.y * W + y;
    if (gx < P.n[k] && gy < P.n[k]) P.p[k][l * P.plane[k] + GIDX(P.pitch[k], gy, gx)] = v;
  }
}

/* what a quad reads of one layer besides its centre: the rows below (up: y-1) and above (dn: y+2), the columns
 * x-1 (w) and x+2 (e), b, and the stretching of the interface below the layer or lambda (s, when s != null) */
struct PyrIn {
  double2 up, dn, b0, b1, s0, s1;
  double w0, w1, e0, e1;
};
__device__ __forceinline__ void pyr_load(PyrIn &L, const double *__restrict__ al, const double *__restrict__ bl,
                                         const double *__restrict__ sl, size_t c0, size_t c1, int W) {
  L.up = *(const double2 *)(al + c0 - W); L.dn = *(const double2 *)(al + c1 + W);
  L.w0 = al[c0 - 1]; L.w1 = al[c1 - 1]; L.e0 = al[c0 + 2]; L.e1 = al[c1 + 2];
  L.b0 = *(const double2 *)(bl + c0); L.b1 = *(const double2 *)(bl + c1);
  if (sl) { L.s0 = *(const double2 *)(sl + c0); L.s1 = *(const double2 *)(sl + c1); }
  else L.s0 = L.s1 = make_double2(0., 0.);
}

template <int NL, bool SFIELD>
__global__ void __launch_bounds__(256, NL <= 8 ? 2 : 1)
k_residual_pyr(const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ res,
               const double *__restrict__ s, StretchConsts S, Geom g, LayerMetrics M, PyrLevels P,
               double *__restrict__ maxres) {
  __shared__ double s2[NL * 64], s3[NL * 16], s4[NL * 4];
  const int lane = threadIdx.x, tid = threadIdx.y * 32 + lane;
  const int qx = blockIdx.x * (PYR_TILE / 2) + (lane & 15);
  const int qy = blockIdx.y * (PYR_TILE / 2) + threadIdx.y * 2 + (lane >> 4);
  const bool in = 2 * qx < g.nx && 2 * qy < g.ny;
  const int W = g.pitch;
  const size_t c0 = GIDX(W, 2 * qy, 2 * qx), c1 = c0 + W;
  const double D = g.Delta, rD = g.rD;
  /* centre rows of the quad, two layers ahead; the rest of a layer's inputs (neighbours, b, stretching or lambda) one
     layer ahead, so that the loads of the next layer are in flight while this one is computed */
  double2 ctr0[NL], ctr1[NL];
  PyrIn ld[NL];
  const bool sfield = NL == 1 || SFIELD;
  if (in) {
    ctr0[0] = *(const double2 *)(a + c0);
    ctr1[0] = *(const double2 *)(a + c1);
    if (NL > 1) {
      ctr0[NL > 1 ? 1 : 0] = *(const double2 *)(a + g.plane + c0);
      ctr1[NL > 1 ? 1 : 0] = *(const double2 *)(a + g.plane + c1);
    }
    pyr_load(ld[0], a, b, sfield ? s : nullptr, c0, c1, W);
  }
  double m = 0.;
#pragma unroll
  for (int l = 0; l < NL; l++) {
    double r00 = 0., r10 = 0., r01 = 0., r11 = 0.; /* r<dx><dy> */
    if (in) {
      const int ln = l + 1 < NL ? l + 1 : l, ln2 = l + 2 < NL ? l + 2 : l;
      if (l + 1 < NL)
        pyr_load(ld[ln], a + ln * g.plane, b + ln * g.plane, sfield && ln < NL - 1 ? s + ln * g.plane : nullptr, c0, c1, W);
      if (l + 2 < NL) {
        ctr0[ln2] = *(const double2 *)(a + ln2 * g.plane + c0);
        ctr1[ln2] = *(const double2 *)(a + ln2 * g.plane + c1);
      }
      const PyrIn &L = ld[l];
      const double2 C0 = ctr0[l], C1 = ctr1[l];
      const int lm = l > 0 ? l - 1 : 0;
      const double2 M0 = ctr0[lm], M1 = ctr1[lm], P0 = ctr0[ln], P1 = ctr1[ln];
      if (NL == 1) {
        r00 = L.b0.x - L.s0.x * C0.x; r10 = L.b0.y - L.s0.y * C0.y; r01 = L.b1.x - L.s1.x * C1.x; r11 = L.b1.y - L.s1.y * C1.y;
      } else {
        double2 sm0, sm1, sp0, sp1;
        if (SFIELD) { /* interface l-1 was loaded with the layer above */
          sm0 = ld[lm].s0; sm1 = ld[lm].s1; sp0 = L.s0; sp1 = L.s1;
        } else {
          sm0 = sm1 = make_double2(S.s[lm], S.s[lm]);
          sp0 = sp1 = make_double2(S.s[l], S.s[l]);
        }
        r00 = res_vertical<NL>(l, L.b0.x, sm0.x, sp0.x, M0.x, C0.x, P0.x, M);
        r10 = res_vertical<NL>(l, L.b0.y, sm0.y, sp0.y, M0.y, C0.y, P0.y, M);
        r01 = res_vertical<NL>(l, L.b1.x, sm1.x, sp1.x, M1.x, C1.x, P1.x, M);
        r11 = res_vertical<NL>(l, L.b1.y, sm1.y, sp1.y, M1.y, C1.y, P1.y, M);
      }
      r00 = res_laplacian(r00, C0.x, L.w0, C0.y, L.up.x, C1.x, D, rD);
      r10 = res_laplacian(r10, C0.y, C0.x, L.e0, L.up.y, C1.y, D, rD);
      r01 = res_laplacian(r01, C1.x, L.w1, C1.y, C0.x, L.dn.x, D, rD);
      r11 = res_laplacian(r11, C1.y, C1.x, L.e1, C0.y, L.dn.y, D, rD);
      *(double2 *)(res + l * g.plane + c0) = make_double2(r00, r10);
      *(double2 *)(res + l * g.plane + c1) = make_double2(r01, r11);
      double f[4] = {fabs(r00), fabs(r10), fabs(r01), fabs(r11)};
#pragma unroll
      for (int i = 0; i < 4; i++) {
        if (NL == 1 && !(f[i] > 0.)) f[i] = 0.; /* k_residual_scalar maps NaN to 0, k_residual skips it */
        if (f[i] > m) m = f[i];
      }
    }
    if (P.nlev >= 1) {
      const double v1 = restrict4(r00, r01, r10, r11);
      if (in) P.p[0][l * P.plane[0] + GIDX(P.pitch[0], qy, qx)] = v1;
      if (P.nlev >= 2) {
        const double u01 = __shfl_down_sync(FULLMASK, v1, 16), u10 = __shfl_down_sync(FULLMASK, v1, 1),
                     u11 = __shfl_down_sync(FULLMASK, v1, 17);
        if (lane < 16 && !(lane & 1)) {
          const double v2 = restrict4(v1, u01, u10, u11);
          if (in) P.p[1][l * P.plane[1] + GIDX(P.pitch[1], qy >> 1, qx >> 1)] = v2;
          s2[(l * 8 + threadIdx.y) * 8 + (lane >> 1)] = v2;
        }
      }
    }
  }
  if (P.nlev >= 3) {
    __syncthreads();
    pyr_stage<NL, 4>(s2, s3, P, 2, tid);
    if (P.nlev >= 4) {
      __syncthreads();
      pyr_stage<NL, 2>(s3, s4, P, 3, tid);
      if (P.nlev >= 5) {
        __syncthreads();
        pyr_stage<NL, 1>(s4, nullptr, P, 4, tid);
      }
    }
  }
  block_max_to(maxres, m);
}

/* [BASILISK] poisson.h residual(), scalar Helmholtz, lambda field:
 *   res = b - lambda*a + face-gradient form as above */
__global__ void __launch_bounds__(256)
k_residual_scalar(const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ res,
                  const double *__restrict__ lam, Geom g, double *__restrict__ maxres) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  double m = 0.;
  if (x < g.nx && y < g.ny) {
    const size_t c = GIDX(g.pitch, y, x);
    const double D = g.Delta, rD = g.rD;
    const double ac = a[c];
    const double r = res_laplacian(b[c] - lam[c] * ac, ac, a[c - 1], a[c + 1], a[c - g.pitch], a[c + g.pitch], D, rD);
    res[c] = r;
    m = fabs(r);
    if (!(m > 0.)) m = 0.;
  }
  block_max_to(maxres, m);
}

/* ------------------------------------------------------------------ restriction
 * [BASILISK] restriction_average: sum over foreach_child() in the order
 * (x,y) = (0,0),(0,1),(1,0),(1,1), then /4.  gc = coarse geometry. */
__global__ void k_restrict(const double *__restrict__ fine, double *__restrict__ coarse, Geom gf, Geom gc,
                           double sg, int write_ghosts) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= gc.nx || y >= gc.ny) return;
  const double *a = fine + (size_t)f * gf.plane;
  const size_t c00 = GIDX(gf.pitch, 2 * y, 2 * x);
  double sum = 0.;
  sum += a[c00];
  sum += a[c00 + gf.pitch];
  sum += a[c00 + 1];
  sum += a[c00 + gf.pitch + 1];
  const double v = sum / 4;
  double *cp = coarse + (size_t)f * gc.plane;
  cp[GIDX(gc.pitch, y, x)] = v;
  if (write_ghosts) {
    const int nx = gc.nx, ny = gc.ny;
    const bool l = x == 0, r = x == nx - 1, bo = y == 0, t = y == ny - 1;
    if (l) cp[GIDX(gc.pitch, y, -1)] = sg * v;
    if (r) cp[GIDX(gc.pitch, y, nx)] = sg * v;
    if (bo) cp[GIDX(gc.pitch, -1, x)] = sg * v;
    if (t) cp[GIDX(gc.pitch, ny, x)] = sg * v;
    if (l && bo) cp[GIDX(gc.pitch, -1, -1)] = v;
    if (l && t) cp[GIDX(gc.pitch, ny, -1)] = v;
    if (r && bo) cp[GIDX(gc.pitch, -1, nx)] = v;
    if (r && t) cp[GIDX(gc.pitch, ny, nx)] = v;
  }
}

/* ------------------------------------------------------------------ prolongation
 * [BASILISK] bilinear(): (9*C + 3*(C[cx,0] + C[0,cy]) + C[cx,cy])/16 with the
 * coarse ghost ring of a homogeneous-dirichlet `da` evaluated on the fly
 * (ghost = -mirror, corner = +mirror), so da ghosts are never stored. */
__device__ __forceinline__ double coarse_at(const double *__restrict__ c, const Geom &gc, int x, int y) {
  double s = 1.;
  /* physical side: homogeneous-dirichlet ghost by reflection; internal side: stored halo value */
  if (x < 0) { if (!(gc.bc & 1)) { x = 0; s = -s; } } else if (x >= gc.nx) { if (!(gc.bc & 2)) { x = gc.nx - 1; s = -s; } }
  if (y < 0) { if (!(gc.bc & 4)) { y = 0; s = -s; } } else if (y >= gc.ny) { if (!(gc.bc & 8)) { y = gc.ny - 1; s = -s; } }
  return s * c[GIDX(gc.pitch, y, x)];
}

__global__ void k_prolong(const double *__restrict__ coarse, double *__restrict__ fine, Geom gc, Geom gf) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= gf.nx || y >= gf.ny) return;
  const double *c = coarse + (size_t)f * gc.plane;
  const int xc = x >> 1, yc = y >> 1;
  const int cx = (x & 1) ? 1 : -1, cy = (y & 1) ? 1 : -1;
  const double v = (9. * coarse_at(c, gc, xc, yc) +
                    3. * (coarse_at(c, gc, xc + cx, yc) + coarse_at(c, gc, xc, yc + cy)) +
                    coarse_at(c, gc, xc + cx, yc + cy)) / 16.;
  fine[(size_t)f * gf.plane + GIDX(gf.pitch, y, x)] = v;
}

/* Same operator, one thread per COARSE cell: the 3x3 coarse neighbourhood is read once and the four
 * children are written as two 16-byte stores (the per-child kernel above re-reads it four times and is
 * instruction-bound: ncu, profiles/r01_ncu_kernels.md).  Needs even fine tile sizes aligned with the
 * coarse cells (always true on one GPU). */
__global__ void __launch_bounds__(256)
k_prolong4(const double *__restrict__ coarse, double *__restrict__ fine, Geom gc, Geom gf) {
  const int xc = blockIdx.x * blockDim.x + threadIdx.x;
  const int yc = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (xc >= gc.nx || yc >= gc.ny) return;
  const double *c = coarse + (size_t)f * gc.plane;
  double v[3][3];
  if (xc > 0 && xc < gc.nx - 1 && yc > 0 && yc < gc.ny - 1) {
    const double *p = c + GIDX(gc.pitch, yc, xc);
#pragma unroll
    for (int dy = 0; dy < 3; dy++)
#pragma unroll
      for (int dx = 0; dx < 3; dx++) v[dy][dx] = p[(dy - 1) * gc.pitch + (dx - 1)];
  } else {
#pragma unroll
    for (int dy = 0; dy < 3; dy++)
#pragma unroll
      for (int dx = 0; dx < 3; dx++) v[dy][dx] = coarse_at(c, gc, xc + dx - 1, yc + dy - 1);
  }
  double *o = fine + (size_t)f * gf.plane + GIDX(gf.pitch, 2 * yc, 2 * xc);
#pragma unroll
  for (int oy = 0; oy < 2; oy++) {
    double r[2];
#pragma unroll
    for (int ox = 0; ox < 2; ox++) {
      const int ix = ox ? 2 : 0, iy = oy ? 2 : 0;
      r[ox] = (9. * v[1][1] + 3. * (v[1][ix] + v[iy][1]) + v[iy][ix]) / 16.;
    }
    *reinterpret_cast<double2 *>(o + (size_t)oy * gf.pitch) = make_double2(r[0], r[1]);
  }
}

/* ------------------------------------------------------------------ wavelet transform
 * [BASILISK] wavelet() / inverse_wavelet() (grid/multigrid-common.h) for the multi-scale filter of msqg
 * (wavelet_filter, msqg/qg.h:509-560): the coefficient of a fine cell is its value minus the bilinear
 * prolongation of the restricted field; the filter multiplies it by sig_lev (qg.h:533-537, fused here).
 * One thread per coarse cell and layer (blockIdx.z), four children; the field has homogeneous dirichlet
 * boundaries (psi), evaluated on the fly like in k_prolong. */
template <bool INVERSE>
__global__ void __launch_bounds__(256)
k_wavelet(const double *__restrict__ sc, double *__restrict__ sf, double *__restrict__ wf, const double *__restrict__ sig,
          Geom gc, Geom gf, int write_ghosts) {
  const int xc = blockIdx.x * blockDim.x + threadIdx.x;
  const int yc = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (xc >= gc.nx || yc >= gc.ny) return;
  const double *c = sc + (size_t)f * gc.plane;
  double v[3][3];
#pragma unroll
  for (int dy = 0; dy < 3; dy++)
#pragma unroll
    for (int dx = 0; dx < 3; dx++) v[dy][dx] = coarse_at(c, gc, xc + dx - 1, yc + dy - 1);
#pragma unroll
  for (int oy = 0; oy < 2; oy++)
#pragma unroll
    for (int ox = 0; ox < 2; ox++) {
      const int ix = ox ? 2 : 0, iy = oy ? 2 : 0;
      const double sp = (9. * v[1][1] + 3. * (v[1][ix] + v[iy][1]) + v[iy][ix]) / 16.;
      const int x = 2 * xc + ox, y = 2 * yc + oy;
      const size_t o = (size_t)f * gf.plane + GIDX(gf.pitch, y, x);
      if (!INVERSE) {
        double w = sf[o];
        w -= sp; /* difference between fine value and its prolongation */
        w *= sig[GIDX(gf.pitch, y, x)];
        wf[o] = w;
      } else {
        double s = sp;
        s += wf[o];
        sf[o] = s;
        if (write_ghosts) {
          double *p = sf + (size_t)f * gf.plane;
          const bool l = x == 0, r = x == gf.nx - 1, bo = y == 0, t = y == gf.ny - 1;
          if (l) p[GIDX(gf.pitch, y, -1)] = -s;
          if (r) p[GIDX(gf.pitch, y, gf.nx)] = -s;
          if (bo) p[GIDX(gf.pitch, -1, x)] = -s;
          if (t) p[GIDX(gf.pitch, gf.ny, x)] = -s;
          if (l && bo) p[GIDX(gf.pitch, -1, -1)] = s;
          if (l && t) p[GIDX(gf.pitch, gf.ny, -1)] = s;
          if (r && bo) p[GIDX(gf.pitch, -1, gf.nx)] = s;
          if (r && t) p[GIDX(gf.pitch, gf.ny, gf.nx)] = s;
        }
      }
    }
}
/* root cell: w = s*sig_lev (forward + filter), s = w (inverse); level 0 is one cell per layer */
__global__ void k_wavelet_root(double *__restrict__ s0, double *__restrict__ w0, Geom g0, double sig0, int nf, int inverse) {
  const int f = threadIdx.x;
  if (f >= nf) return;
  const size_t o = (size_t)f * g0.plane + GIDX(g0.pitch, 0, 0);
  if (!inverse) { double w = s0[o]; w *= sig0; w0[o] = w; }
  else s0[o] = w0[o];
}
/* qof = (qof*nbar + (tmp - qo)/dtflt)/(nbar+1) + boundary(qofl), qg.h:543-557 */
__global__ void k_filter_mean(double *__restrict__ qof, const double *__restrict__ tmp, const double *__restrict__ qo, Geom g,
                              double dtflt, int nbar) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= g.nx || y >= g.ny) return;
  const size_t c = (size_t)f * g.plane + GIDX(g.pitch, y, x);
  const double v = (qof[c] * nbar + (tmp[c] - qo[c]) / dtflt) / (nbar + 1);
  qof[c] = v;
  double *p = qof + (size_t)f * g.plane;
  const bool l = x == 0, r = x == g.nx - 1, bo = y == 0, t = y == g.ny - 1;
  if (l) p[GIDX(g.pitch, y, -1)] = -v;
  if (r) p[GIDX(g.pitch, y, g.nx)] = -v;
  if (bo) p[GIDX(g.pitch, -1, x)] = -v;
  if (t) p[GIDX(g.pitch, g.ny, x)] = -v;
  if (l && bo) p[GIDX(g.pitch, -1, -1)] = v;
  if (l && t) p[GIDX(g.pitch, g.ny, -1)] = v;
  if (r && bo) p[GIDX(g.pitch, -1, g.nx)] = v;
  if (r && t) p[GIDX(g.pitch, g.ny, g.nx)] = v;
}
/* filter_de, qg_energy.h:214-224: de_ft += tmp*dtflt*(-pm*(1-ediag)+ediag); pm = 0 */
__global__ void k_filter_de(double *__restrict__ de_ft, const double *__restrict__ tmp2, double *__restrict__ pm, Geom g,
                            double dtflt, double ediag) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= g.nx || y >= g.ny) return;
  const size_t c = (size_t)f * g.plane + GIDX(g.pitch, y, x);
  de_ft[c] += tmp2[c] * dtflt * (-pm[c] * (1 - ediag) + ediag);
  pm[c] = 0;
}

/* ------------------------------------------------------------------ correction
 * mg_cycle tail: a += da ; boundary(a)   (mspg/elliptic.h:92-98).  Ghost ring of
 * the dirichlet(0) field a is written by the boundary cells themselves. */
__global__ void k_correct(double *__restrict__ a, const double *__restrict__ da, Geom g, int phys_only = 0) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= g.nx || y >= g.ny) return;
  double *ap = a + (size_t)f * g.plane;
  const size_t c = GIDX(g.pitch, y, x);
  const double v = ap[c] + da[(size_t)f * g.plane + c];
  ap[c] = v;
  const int nx = g.nx, ny = g.ny;
  /* phys_only: ghosts of the PHYSICAL sides only (red-black tiles keep the neighbour's cells in the ring of an internal
     side and correct them in place, k_correct_ring); otherwise all four sides, the halo exchange that follows overwrites
     the internal ones */
  const int ib = phys_only ? g.bc : 0;
  const bool l = x == 0 && !(ib & 1), r = x == nx - 1 && !(ib & 2), bo = y == 0 && !(ib & 4), t = y == ny - 1 && !(ib & 8);
  if (l) ap[GIDX(g.pitch, y, -1)] = -v;
  if (r) ap[GIDX(g.pitch, y, nx)] = -v;
  if (bo) ap[GIDX(g.pitch, -1, x)] = -v;
  if (t) ap[GIDX(g.pitch, ny, x)] = -v;
  if (l && bo) ap[GIDX(g.pitch, -1, -1)] = v;
  if (l && t) ap[GIDX(g.pitch, ny, -1)] = v;
  if (r && bo) ap[GIDX(g.pitch, -1, nx)] = v;
  if (r && t) ap[GIDX(g.pitch, ny, nx)] = v;
}

/* ------------------------------------------------------------------ relax_layer
 * Lexicographic Gauss-Seidel in the reference's traversal order (x outer,
 * y inner, [BASILISK] foreach_level) with the per-column Thomas solve of
 * msqg/poisson_layer.h:80-146, nsweeps sweeps (each followed by the homogeneous
 * dirichlet boundary_level of mg_cycle, mspg/elliptic.h:83-86) fused in ONE
 * pipelined wavefront pass:
 *
 *   - a warp ("worker" w) owns a strip of W = 32/K columns; its 32 lanes are K
 *     sweep groups x W column slots: lane (k,c) applies sweep k to column
 *     i = w*W + c - k.  Shifting the strip left by one column per sweep keeps
 *     the east dependency (sweep k-1, column i+1) inside the warp, so workers
 *     form a one-directional chain w-1 -> w.
 *   - lane (k,c) handles row j = tau - c - 2k - 1 at step tau.  All neighbour
 *     values are warp shuffles of the results the lanes hold at the top of a
 *     step (= what they computed in step tau-1):
 *       west  (sweep k,   i-1, j)   <- lane-1,   used in this step (critical path)
 *       south (sweep k,   i,   j-1) =  own previous result
 *       east  (sweep k-1, i+1, j)   <- lane-W,   used in the NEXT step
 *       north (sweep k-1, i,   j+1) <- lane-W-1, used in the NEXT step
 *     (sweep groups lag each other by two steps, which takes east/north off the
 *     critical path.)  Sweep 0 reads east/north from the initial iterate,
 *     streamed from HBM into a shared-memory row ring with cp.async a fixed
 *     number of rows ahead; res streams the same way.
 *   - the west column of a strip comes from the neighbouring worker through a
 *     global-memory mailbox whose entries are self-validating (a reserved NaN
 *     payload means "not yet written"), so no flags or fences are needed; the
 *     consumer prefetches the next entry one step ahead and re-arms what it
 *     read.
 *   - dirichlet ghosts are evaluated as -(pre-sweep centre value), exactly what
 *     boundary_level left in the ghost ring before the sweep.
 *   - only the last sweep's values are stored: HBM sees one read of da/res and
 *     one write of da for all nsweeps sweeps.
 *
 * A step is latency-bound by the Thomas recurrence (~50 dependent fp64 ops,
 * ~8 cycles each); the loop body is one basic block (plus rare slow paths) so
 * that loads, stores, streaming and mailbox traffic issue in the shadow of
 * that chain.  The Thomas pivots do not depend on the iterate; for horizontally uniform
 * stretching they are per-level constants computed on the host with the
 * reference's expression order (RelaxCoef), and divisions by them use
 * div_by().  Every worker waits only on its left neighbour; the kernel is
 * launched cooperatively so all workers are resident.  Spins are bounded.
 */
template <int NL>
struct RelaxCoef {
  double t0[NL], t2[NL], t1p[NL], rinv[NL]; /* t1p: pivots after forward elimination */
  double cf[NL], cb[NL];                    /* RN(t0[l]*rinv[l-1]), RN(t2[l]*rinv[l]): quotient estimates of k_relax_ws */
  double msd2;                              /* -sq(Delta) */
};

struct RelaxArgs {
  double *da;        /* in/out, level planes [NL] */
  const double *res; /* rhs of the correction equation */
  Geom g;
  int nsweeps;                  /* 1..K */
  unsigned long long *mailbox;  /* [nworkers][K][n][NLP] words, armed with MAIL_EMPTY */
  int *err;                     /* set to 1 on spin timeout */
  long long *dbg;               /* optional [nworkers][4]: start ns, end ns, spins, - */
  int unused;                   /* keeps the struct at 160 bytes, so that the RelaxCoef argument after it starts 16-byte
                                   aligned in the kernel's parameter space: ptxas then loads coefficient pairs with
                                   128-bit constant loads (LDCU.128) */
  const double *rowcoef;        /* k_relax_ws<..., RCOEF>: [ny][6][NL] per-row t0, t2, t1p, rinv, cf, cb (stretching varies with y) */
  int coef_cell;                /* 1: the table is per cell, [ny][nx][6][NL] (stretching varies with x too: frpg_*.bas, qg.h:957-962) */
  int w_base;                   /* k_relax_ws: index of the first strip of this launch (levels wider than the device holds
                                   co-resident strips are swept in column panels; the mailbox carries the boundary column) */
};

#define MAIL_EMPTY 0xFFF8DEADBEEF0001ull
#define SPIN_LIMIT (1 << 22)

__device__ __forceinline__ void cp_async8_if(bool p, unsigned smem_addr, const void *gsrc) {
  asm volatile("{\n .reg .pred q;\n setp.ne.b32 q, %0, 0;\n @q cp.async.ca.shared.global [%1], [%2], 8;\n}\n"
               ::"r"((int)p), "r"(smem_addr), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }
__device__ __forceinline__ void ld_mail2_if(bool p, const unsigned long long *a, unsigned long long &v0,
                                            unsigned long long &v1) {
  asm volatile("{\n .reg .pred q;\n setp.ne.b32 q, %2, 0;\n @q ld.volatile.global.v2.u64 {%0, %1}, [%3];\n}\n"
               : "+l"(v0), "+l"(v1) : "r"((int)p), "l"(a));
}
__device__ __forceinline__ void st_mail2_if(bool p, unsigned long long *a, unsigned long long v0, unsigned long long v1) {
  asm volatile("{\n .reg .pred q;\n setp.ne.b32 q, %0, 0;\n @q st.global.cg.v2.u64 [%1], {%2, %3};\n}\n"
               ::"r"((int)p), "l"(a), "l"(v0), "l"(v1) : "memory");
}

/* Per-row Thomas coefficients of one level for stretching that varies with y only (varRo > 0): the expressions
 * of relax_coef_layers() (msqg/poisson_layer.h:89-139, same order, IEEE division) evaluated with the level's
 * restricted stretching field at column 0 of every row.  out[j][6][NL] = t0, t2, t1p, rinv, cf, cb. */
template <int NL>
__global__ void k_rowcoef(const double *__restrict__ s, Geom g, LayerMetrics M, double *__restrict__ out, int cell) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; /* one thread per row, or per cell (x fastest) */
  if (t >= (size_t)g.ny * (cell ? g.nx : 1)) return;
  const int j = cell ? (int)(t / g.nx) : (int)t, ix = cell ? (int)(t % g.nx) : 0;
  const double D2 = g.Delta * g.Delta;
  double sv[NL], t0[NL], t1[NL], t2[NL];
#pragma unroll
  for (int l = 0; l < NL; l++) { sv[l] = (l < NL - 1) ? s[(size_t)l * g.plane + GIDX(g.pitch, j, ix)] : 0.; t0[l] = t1[l] = t2[l] = 0.; }
  if (NL > 1) {
    t2[0] = -D2 * sv[0] * M.idh1[0];
    t1[0] = -t2[0];
    t1[0] += 1. + 1.; t1[0] += 1. + 1.;
#pragma unroll
    for (int l = 1; l < NL - 1; l++) {
      t0[l] = -D2 * sv[l - 1] * M.idh0[l];
      t2[l] = -D2 * sv[l] * M.idh1[l];
      t1[l] = -t0[l] - t2[l];
      t1[l] += 1. + 1.; t1[l] += 1. + 1.;
    }
    t0[NL - 1] = -D2 * sv[NL - 2] * M.idh0[NL - 1];
    t1[NL - 1] = -t0[NL - 1];
    t1[NL - 1] += 1. + 1.; t1[NL - 1] += 1. + 1.;
#pragma unroll
    for (int l = 1; l < NL; l++) t1[l] -= t0[l] * t2[l - 1] / t1[l - 1];
  }
  double *o = out + t * 6 * NL;
#pragma unroll
  for (int l = 0; l < NL; l++) {
    const double r = 1. / t1[l];
    o[0 * NL + l] = t0[l]; o[1 * NL + l] = t2[l]; o[2 * NL + l] = t1[l]; o[3 * NL + l] = r;
    o[4 * NL + l] = l > 0 ? t0[l] * (1. / t1[l - 1]) : 0.;
    o[5 * NL + l] = t2[l] * r;
  }
}

/* The same table for ONE vertical mode whose lambda = iBu is a field (horizontally varying Fr/Ro, eigmode.h:257-266):
 * the scalar relaxation divides by d = -lambda[]*sq(Delta) + 2 + 2 ([BASILISK] poisson.h relax(), in-tree copy
 * mspg/elliptic.h:294-301), accumulated per dimension as the reference does.  out[j][i][6] = 0, 0, d, 1/d, 0, 0 in
 * the layout of k_rowcoef<1> (per cell), read by the RCOEF instances of the NL = 1 relax kernels. */
__global__ void k_modecoef(const double *__restrict__ lam, Geom g, double *__restrict__ out) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)g.ny * g.nx) return;
  const int j = (int)(t / g.nx), ix = (int)(t % g.nx);
  double d = -lam[GIDX(g.pitch, j, ix)] * (g.Delta * g.Delta);
  d += 1. + 1.; d += 1. + 1.;
  double *o = out + t * 6;
  o[0] = 0.; o[1] = 0.; o[2] = d; o[3] = 1. / d; o[4] = 0.; o[5] = 0.;
}

/* ------------------------------------------------------------------ relax_layer, warp-specialised
 * The wavefront and mailbox protocol described above (lane (k,c) does row tau - c - 2k - 1 at step
 * tau), with each strip served by TWO warps so that the warp on the critical
 * path issues little more than the Thomas recurrence:
 *
 *   compute warp C : W shuffle, Thomas solve, results -> shared-memory ring of its sweep;
 *                    east/north of sweep k come from the ring of sweep k-1 (slot c+1 / slot c),
 *                    sweep 0 reads the same way from the ring of the initial iterate, res from
 *                    its own ring; the strip's west column sits in slot 0 of each sweep ring.
 *   helper warp H  : streams da/res rows HBM -> rings (cp.async, L2-prefetched ahead), polls the
 *                    global mailbox of the left neighbour and deposits entries into slot 0,
 *                    re-arms them, drains the last sweep's rows to HBM.
 *
 * H publishes, per sweep, ONE number: the last row whose inputs are complete (streamed rows landed,
 * mailbox row deposited, ring row drained); C loads the inputs of step tau+1 speculatively at the
 * start of step tau, in the shadow of the recurrence, and checks that number afterwards.
 *
 * A step costs (nx + ny) times on the critical path of a sweep, so the dependent chain is kept as
 * short as IEEE-exact arithmetic allows (measured on B200: fp64 add/mul/fma 8.3 cycles, 64-bit
 * shuffle 24, scripts/ubench):
 *   - x/d for the constant pivots d is RN(x/d) by two Newton-Markstein corrections of ANY estimate
 *     q0 that is within a few ulps (div_fix): the first correction makes it faithful, the second
 *     correctly rounded.  The estimate is formed in parallel with x itself from pre-multiplied
 *     constants (cf = t0*r, cb = t2*r, rr = rhs*r), which takes one operation off the chain per
 *     layer in each direction: 6*(NL-1) + 5 + 6*(NL-1) + 3 dependent operations per step.
 *   - every out[l] is shuffled / stored as soon as it exists; only out[0] -> W -> rhs[0] is exposed.
 *   - rings hold layer PAIRS as 16-byte vectors, [row][pair][slot]: a sweep group (quarter warp)
 *     reads consecutive 16-byte slots, so the 128-bit loads are conflict-free.
 *   - rows 0 and ny-1 and the first/last W+2K steps run an EDGE instance of the step (ghost
 *     substitution for south/north); the steady state runs a leaner instance, unrolled twice.
 */
template <int NL, int K>
struct WsCfg {
  static_assert(K == 4 || K == 8, "lanes = K sweeps x 32/K columns");
  static constexpr int W = 32 / K, S = W + 1, RC = W + K - 1;
  static constexpr int RIN = 32, R2 = 16;
  static constexpr int NLP = (NL + 1) & ~1;   /* mailbox entry padded to 16 bytes */
  static constexpr int NV = NLP / 2;          /* 16-byte vectors (layer pairs) per cell */
  static constexpr int DROW = NV * S, RROW = NV * RC; /* ring row, in vectors */
  static constexpr int XRS = R2 * DROW + (K == 8 ? 4 : 0); /* sweep-ring stride (K = 8: two groups per quarter warp, skew the banks) */
  static constexpr int TAIL = W + 2 * K - 2; /* steps after which a streamed row is dead */
  static constexpr int NCNT = 32;            /* ints of counters per worker */
  static constexpr int VECS = RIN * DROW + RIN * RROW + K * XRS + NCNT / 4;
  static constexpr int DOUBLES = 2 * VECS;
  static constexpr size_t smem_per_worker = (size_t)DOUBLES * sizeof(double);
  static constexpr int EPL_D = (NL * S + 31) / 32, EPL_R = (NL * RC + 31) / 32;
  static constexpr int Q = 32 / K; /* mailbox rows polled per sweep per helper iteration */
  enum { C_DONE = 0, H_DONE = 3, LIM = 8, HLIM = 16 }; /* LIM + k: last row jn whose inputs are complete for sweep k */
};
#define WS_INF 0x3fffffff

__device__ __forceinline__ int ld_cnt(const volatile int *p) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared((const void *)p)));
  return v;
}
__device__ __forceinline__ int ld_cnt_a(unsigned a) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void st_cnt_if(bool p, unsigned a, int v) {
  asm volatile("{\n .reg .pred q;\n setp.ne.b32 q, %0, 0;\n @q st.volatile.shared.s32 [%1], %2;\n}\n" ::"r"((int)p), "r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ double2 lds2(unsigned a) {
  double2 v;
  asm volatile("ld.volatile.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts2(unsigned a, double x, double y) {
  asm volatile("st.volatile.shared.v2.f64 [%0], {%1, %2};" ::"r"(a), "d"(x), "d"(y) : "memory");
}
__device__ __forceinline__ double2 lds2_if(bool p, unsigned a) {
  double2 v = make_double2(0., 0.);
  asm volatile("{\n .reg .pred q;\n setp.ne.b32 q, %2, 0;\n @q ld.volatile.shared.v2.f64 {%0, %1}, [%3];\n}\n"
               : "+d"(v.x), "+d"(v.y) : "r"((int)p), "r"(a));
  return v;
}
__device__ __forceinline__ void sts2_if(bool p, unsigned a, double x, double y) {
  asm volatile("{\n .reg .pred q;\n setp.ne.b32 q, %0, 0;\n @q st.volatile.shared.v2.f64 [%1], {%2, %3};\n}\n"
               ::"r"((int)p), "r"(a), "d"(x), "d"(y) : "memory");
}
/* RN(x/d) from any estimate q of x/d that is good to a few ulps; r = RN(1/d) */
__device__ __forceinline__ double div_fix(double x, double q, double d, double r) {
  double e = __fma_rn(-d, q, x);
  q = __fma_rn(e, r, q);
  e = __fma_rn(-d, q, x);
  return __fma_rn(e, r, q);
}

/* One CTA per SM is all the shared-memory rings allow, so say so: without the second argument ptxas budgets 128
 * registers for a 256-thread block (spills 16 bytes in the step loop); with it the kernel takes 146, no spill, and the
 * finest-level launch goes from 3387 to 3304 us (scripts/ubench/relax_bench.cu, same checksum).  WS_MINBLOCKS=0 restores
 * the default budget (A/B measurements). */
#ifndef WS_MINBLOCKS
#define WS_MINBLOCKS 1
#endif
#if WS_MINBLOCKS > 0
#define WS_LAUNCH_BOUNDS(NT) __launch_bounds__(NT, WS_MINBLOCKS)
#else
#define WS_LAUNCH_BOUNDS(NT) __launch_bounds__(NT)
#endif
template <int NL, int K, int WPC, bool TILE, bool RCOEF = false>
__global__ void WS_LAUNCH_BOUNDS(64 * WPC)
k_relax_ws(RelaxArgs A, RelaxCoef<NL> C) {
  constexpr bool MW = false; /* (a dedicated mail warp per CTA was measured slower and has been removed) */
  using Cfg = WsCfg<NL, K>;
  constexpr int W = Cfg::W, S = Cfg::S, RC = Cfg::RC, RIN = Cfg::RIN, R2 = Cfg::R2;
  constexpr int NLP = Cfg::NLP, NV = Cfg::NV, DROW = Cfg::DROW, RROW = Cfg::RROW, XRS = Cfg::XRS, Q = Cfg::Q;
  extern __shared__ double2 smem2[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool mailer = MW && warp == 2 * WPC;
  const bool helper = warp >= WPC && !mailer;
  const int wl = mailer ? 0 : (helper ? warp - WPC : warp); /* worker slot inside the CTA */
  const int nx = A.g.nx, ny = A.g.ny; /* columns / rows of this tile */
  /* internal sides (multi-GPU tiles, single-sweep launches only): ghosts are stored halo values */
  const bool lint = TILE && (A.g.bc & 1), rint = TILE && (A.g.bc & 2), bint = TILE && (A.g.bc & 4), tint = TILE && (A.g.bc & 8);
  const int r_first = bint ? -1 : 0, r_last = tint ? ny : ny - 1; /* rows of the iterate that are streamed */
  /* the same value in every lane; routed through a shuffle because ptxas then keeps the faster schedule of the
     compute loop (676 instead of 703 cycles per step, scripts/ubench/relax_bench.cu) */
  const int w = __shfl_sync(FULLMASK, A.w_base + (int)blockIdx.x * WPC + wl, 0);
  const int nworkers = (nx + K - 1 + W - 1) / W;
  double2 *base = smem2 + (size_t)wl * Cfg::VECS;
  double2 *IN = base;                   /* [RIN][NV][S]  initial iterate, slot s <-> column w*W + s */
  double2 *RES = IN + RIN * DROW;       /* [RIN][NV][RC] rc <-> column w*W - (K-1) + rc */
  double2 *XR = RES + RIN * RROW;       /* K rings [R2][NV][S]: slot 0 west column, slot c+1 lane c */
  volatile int *cnt = (volatile int *)(XR + K * XRS);
  const int nsw = A.nsweeps;
  const int kf = nsw - 1;
  /* slot 2 is unused; it starts at 0 like C_DONE and H_DONE because ptxas schedules the setup differently otherwise */
  if (lane < Cfg::NCNT && !helper && !mailer) cnt[lane] = (lane == Cfg::C_DONE || lane == 2 || lane == Cfg::H_DONE) ? 0 : -1000;
  __syncthreads();
  if (w < nworkers) {
  const int pitch = A.g.pitch;
  const size_t plane = A.g.plane;
  const bool has_consumer = (w + 1 < nworkers);

  if (!helper && !mailer) {
    /* ================================================================ compute warp */
    const int k = lane / W, c = lane % W;
    const int i = w * W + c - k;
    const bool col_ok = (i >= 0 && i < nx && k < nsw);
    const bool k0 = (k == 0);
    const bool left = (i == 0) && !lint, right = (i == nx - 1) && !rint;
    const bool use_mail = (c == 0) && (w > 0 || lint);
    const bool lr_any = __any_sync(FULLMASK, left || right);
    const bool wr_valid = has_consumer && (w * W + W - 1 - k) >= 0 && (w * W + W - 1 - k) < nx;
    /* Neighbouring strips of the SAME CTA hand their boundary column over through shared memory:
       the consumer reads slot W of the producer's sweep rings directly, guarded by the producer's
       step counter (and the producer checks the consumer's counter before it reuses a ring row).
       Only the first strip of a CTA goes through the global mailbox and its helper warp. */
    const bool din = (wl > 0), dout = has_consumer && (wl + 1 < WPC);
    const bool mb_writer = wr_valid && c == W - 1 && col_ok && !dout;
    const bool st_lane = (k < nsw);
    unsigned long long *mo = A.mailbox + ((size_t)w * K + k) * (size_t)ny * NLP; /* + j*NLP */
    /* shared-memory byte addresses */
    const unsigned a_in = (unsigned)__cvta_generic_to_shared(k0 ? IN : XR + (size_t)(k - 1) * XRS) + 16u * c;
    const int in_mask = k0 ? RIN - 1 : R2 - 1;
    const unsigned a_ring = (unsigned)__cvta_generic_to_shared(XR + (size_t)(k < K ? k : 0) * XRS);
    const double2 *XRL = XR - Cfg::VECS; /* sweep rings of the left neighbour in this CTA (din only) */
    /* west column of sweep k: slot 0 of the own ring (mailbox deposits) or slot W of the neighbour's ring */
    const unsigned a_west = din ? (unsigned)__cvta_generic_to_shared(XRL + (size_t)(k < K ? k : 0) * XRS) + 16u * W : a_ring;
    /* north of lane c = 0, sweep k > 0, is the west column of sweep k-1 */
    const unsigned a_north = (din && c == 0 && !k0) ? (unsigned)__cvta_generic_to_shared(XRL + (size_t)(k - 1) * XRS) + 16u * W : a_in;
    const unsigned a_cdp = (unsigned)__cvta_generic_to_shared((const void *)(cnt + Cfg::C_DONE)) - (din ? (unsigned)(Cfg::VECS * 16) : 0u);
    const unsigned a_cdc = (unsigned)__cvta_generic_to_shared((const void *)(cnt + Cfg::C_DONE)) + (dout ? (unsigned)(Cfg::VECS * 16) : 0u);
    const unsigned a_res = (unsigned)__cvta_generic_to_shared(RES) + 16u * (c - k + K - 1);
    const unsigned a_lim = (unsigned)__cvta_generic_to_shared((const void *)(cnt + Cfg::LIM + k));
    const unsigned a_cdone = (unsigned)__cvta_generic_to_shared((const void *)(cnt + Cfg::C_DONE));

    /* The loop is rotated by half a step: iteration tau does the BACK SUBSTITUTION of step tau (row j)
       and then the right-hand side and FORWARD ELIMINATION of step tau+1 (row jn = j+1).
       Why: ptxas schedules a basic block bottom-up (everything as late as its consumers allow).  With
       the block boundary between two steps, every load, ghost substitution, shuffle and store of a step
       is "needed at the block end" and gets bunched after out[0], on the critical path of the next
       step (measured: ~700 cycles per step against a ~400-cycle chain).  With the boundary in the
       middle of the recurrence the consumers of that work (rhs of the next step, its forward
       elimination) sit in the same block, so it lands in the stall slots of the back substitution.
       Loop-carried: rp[] = right-hand side after forward elimination, q0p = quotient estimate of the
       pivot row, ncur[] = raw north values of the row being solved (= pre-sweep centre of the next). */
    double rp[NL], ncur[NL], q0p = 0.;
#pragma unroll
    for (int l = 0; l < NL; l++) rp[l] = ncur[l] = 0.;
    /* RCOEF (varRo > 0: Ro and with it the stretching depend on y, msqg/qg.h:1032-1048): the Thomas coefficients
       are per-row constants read from a table; cj = row j (back substitution), cn = row jn (forward elimination) */
    constexpr int NCF = RCOEF ? 6 * NL : 2;
    double cj[NCF];
#pragma unroll
    for (int i = 0; i < NCF; i++) cj[i] = 1.;
    long long t_start = 0, n_spins = 0;
    if (A.dbg) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
    const int T = ny + W + 2 * K - 2;

    /* EDGE: rows 0 / ny-1 may occur (ghost substitution for south/north, partial stores); LR: some
       lane of the warp sits on a physical left/right boundary (MODE) */
    auto step = [&](auto edge_tag, auto lr_tag, const int tau) {
      constexpr bool EDGE = decltype(edge_tag)::value;
      constexpr int MODE = decltype(lr_tag)::value; /* 0 interior strip, 1 leftmost strip (no mailbox), 2 general */
      const int j = tau - c - 2 * k - 1;
      const int jn = j + 1;
      /* ---- (B) inputs of step tau+1 (row jn), speculatively; the guard is read first */
      const int lim = ld_cnt_a(a_lim);
      const int cdp = ld_cnt_a(a_cdp), cdc = ld_cnt_a(a_cdc); /* neighbours' step counters (own counter if not direct) */
      double2 e2[NV], n2[NV], b2[NV], w2[NV], s2[NV];
      auto load_inputs = [&]() {
        const unsigned pe = a_in + 16u * (unsigned)((jn & in_mask) * DROW + 1);
        const unsigned pn = a_north + 16u * (unsigned)(((jn + 1) & in_mask) * DROW);
        const unsigned pb = a_res + 16u * (unsigned)((jn & (RIN - 1)) * RROW);
        const unsigned pw = a_west + 16u * (unsigned)((jn & (R2 - 1)) * DROW);
#pragma unroll
        for (int v = 0; v < NV; v++) {
          e2[v] = lds2(pe + 16u * (v * S));
          n2[v] = lds2(pn + 16u * (v * S));
          b2[v] = lds2(pb + 16u * (v * RC));
          if (MODE != 1) w2[v] = lds2_if(use_mail, pw + 16u * (v * S));
          else w2[v] = make_double2(0., 0.);
          if (EDGE && TILE) s2[v] = lds2(a_in + 16u * (unsigned)(((-1) & in_mask) * DROW + v * S)); /* stored halo row -1 */
          else s2[v] = make_double2(0., 0.);
        }
      };
      load_inputs();
      double cn[NCF];
      if (RCOEF) {
        const int rn = min(max(jn, 0), ny - 1);
        const size_t ce = A.coef_cell ? (size_t)rn * nx + min(max(i, 0), nx - 1) : (size_t)rn;
        const double2 *pc = reinterpret_cast<const double2 *>(A.rowcoef + ce * (6 * NL));
        if (A.coef_cell) { /* per-cell tables stream from HBM: pull the lines of this lane's cell 12 rows ahead into L2 */
          const char *pf = reinterpret_cast<const char *>(A.rowcoef + ((size_t)min(rn + 12, ny - 1) * nx + min(max(i, 0), nx - 1)) * (6 * NL));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(pf + 128));
        }
#pragma unroll
        for (int i = 0; i < NCF / 2; i++) { const double2 t = __ldg(pc + i); cn[2 * i] = t.x; cn[2 * i + 1] = t.y; }
      }
      auto T2j = [&](int l) { return RCOEF ? cj[(1 * NL + l) % NCF] : C.t2[l]; };
      auto T1j = [&](int l) { return RCOEF ? cj[(2 * NL + l) % NCF] : C.t1p[l]; };
      auto RIj = [&](int l) { return RCOEF ? cj[(3 * NL + l) % NCF] : C.rinv[l]; };
      auto CBj = [&](int l) { return RCOEF ? cj[(5 * NL + l) % NCF] : C.cb[l]; };
      auto T0n = [&](int l) { return RCOEF ? cn[(0 * NL + l) % NCF] : C.t0[l]; };
      auto T1n = [&](int l) { return RCOEF ? cn[(2 * NL + l) % NCF] : C.t1p[l]; };
      auto RIn = [&](int l) { return RCOEF ? cn[(3 * NL + l) % NCF] : C.rinv[l]; };
      auto CFn = [&](int l) { return RCOEF ? cn[(4 * NL + l) % NCF] : C.cf[l]; };
      /* ---- (C) back substitution of step tau (msqg/poisson_layer.h:141-146); results leave as they appear */
      const unsigned po = a_ring + 16u * (unsigned)((j & (R2 - 1)) * DROW + c + 1);
      const bool row_ok = EDGE ? ((unsigned)j < (unsigned)ny) : true;
      const bool do_st = row_ok && st_lane;
      const bool do_mb = row_ok && mb_writer;
      unsigned long long *mrow = mo + (long long)j * NLP;
      double out[NL], wsh[NL];
      if (NL == 1) out[0] = div_by(rp[0], T1j(0), RIj(0));
      else out[NL - 1] = div_fix(rp[NL - 1], q0p, T1j(NL - 1), RIj(NL - 1));
#pragma unroll
      for (int l = NL - 1; l >= 0; l--) {
        if (l < NL - 1) {
          const double rr = rp[l] * RIj(l);
          const double m = T2j(l) * out[l + 1];
          const double q0 = __fma_rn(-CBj(l), out[l + 1], rr);
          const double x = rp[l] - m;
          out[l] = div_fix(x, q0, T1j(l), RIj(l));
        }
        wsh[l] = __shfl_up_sync(FULLMASK, out[l], 1);
        if ((l & 1) == 0) { /* layer pair (l, l+1) complete */
          const double hi = (l + 1 < NL) ? out[l + 1 < NL ? l + 1 : l] : 0.;
          sts2_if(do_st, po + 16u * ((l >> 1) * S), out[l], hi);
          st_mail2_if(do_mb, mrow + l, (unsigned long long)__double_as_longlong(out[l]), (unsigned long long)__double_as_longlong(hi));
        }
      }
      /* results of step tau are in the rings: publish (helper: drain / ring reuse; right neighbour: hand-off) */
      __syncwarp();
      st_cnt_if(lane == 0, a_cdone, tau + 1);
      /* ---- (D) step tau+1: right-hand side r = -sq(Delta)*b; r += E + W; r += N + S (reference association
         order, msqg/poisson_layer.h:88-94) and forward elimination (:137-140) */
      double cold[NL];
#pragma unroll
      for (int l = 0; l < NL; l++) cold[l] = ncur[l];
      auto next_forward = [&]() {
        double rhs[NL];
#pragma unroll
        for (int l = 0; l < NL; l++) {
          const double ev = (l & 1) ? e2[l >> 1].y : e2[l >> 1].x;
          const double nv = (l & 1) ? n2[l >> 1].y : n2[l >> 1].x;
          const double bv = (l & 1) ? b2[l >> 1].y : b2[l >> 1].x;
          const double wv = (l & 1) ? w2[l >> 1].y : w2[l >> 1].x;
          const double sv = (l & 1) ? s2[l >> 1].y : s2[l >> 1].x;
          /* dirichlet ghost: -(pre-sweep centre of the cell of step tau+1); sign flip on the integer pipe */
          const double g = __hiloint2double(__double2hiint(cold[l]) ^ 0x80000000, __double2loint(cold[l]));
          double aw, ae, as, an;
          if (MODE == 2) { const double alt = left ? g : wv; aw = (left || use_mail) ? alt : wsh[l]; ae = right ? g : ev; }
          else if (MODE == 1) { aw = left ? g : wsh[l]; ae = ev; }
          else { aw = use_mail ? wv : wsh[l]; ae = ev; }
          if (EDGE) { as = (jn == 0) ? ((TILE && bint) ? sv : g) : out[l]; an = (jn == ny - 1 && !tint) ? g : nv; }
          else { as = out[l]; an = nv; }
          double r = C.msd2 * bv;
          r += ae + aw;
          r += an + as;
          rhs[l] = r;
          ncur[l] = nv;
        }
        if (NL > 1) {
          double q = 0.;
#pragma unroll
          for (int l = 1; l < NL; l++) {
            const double x = T0n(l) * rhs[l - 1];
            const double q0 = rhs[l - 1] * CFn(l);
            q = div_fix(x, q0, T1n(l - 1), RIn(l - 1));
            if (l < NL - 1) rhs[l] -= q;
          }
          const double rr = rhs[NL - 1] * RIn(NL - 1); /* off the chain: rhs before elimination */
          q0p = __fma_rn(-q, RIn(NL - 1), rr);
          rhs[NL - 1] -= q;
        }
#pragma unroll
        for (int l = 0; l < NL; l++) rp[l] = rhs[l];
      };
      next_forward();
      /* ---- (E) was the speculation of (B) valid? */
      /* left neighbour (direct): its lane (k, W-1) must have stored row jn of sweep k: counter >= tau + W + 1;
         right neighbour (direct): must be done with the ring row that iteration tau+1 overwrites */
      const int need_p = din ? min(tau + W + 1, T) : -WS_INF, need_c = dout ? tau - R2 - W + 4 : -WS_INF; /* T: the neighbour's final count */
      if (!__all_sync(FULLMASK, jn <= lim && cdp >= need_p && cdc >= need_c)) {
        int spins = 0;
        while (!__all_sync(FULLMASK, jn <= ld_cnt_a(a_lim) && ld_cnt_a(a_cdp) >= need_p && ld_cnt_a(a_cdc) >= need_c)) {
          if (++spins > SPIN_LIMIT) { if (lane == 0) *A.err = 1; break; }
        }
        n_spins += spins;
        __syncwarp();
        load_inputs();
        next_forward();
      }
      if (RCOEF) {
#pragma unroll
        for (int i = 0; i < NCF; i++) cj[i] = cn[i];
      }
    };

    auto run = [&](auto lr_tag) {
      int tau = -1; /* iteration -1 only loads: the pre-sweep value of row 0 is the ghost source of the first row */
      const int t_fast0 = min(T, W + 2 * K - 2), t_fast1 = ny - 2; /* FAST iterations [t_fast0, t_fast1]: every lane has 0 <= j, jn < ny-1 */
#pragma unroll 1
      for (; tau < t_fast0; tau++) step(std::true_type{}, lr_tag, tau);
#pragma unroll 1
#ifndef WS_UNROLL
#define WS_UNROLL 1 /* steady-state steps per loop iteration: 1 / 2 / 3 / 4 measured 3262 / 3290 / 3285 / 3299 us per finest launch */
#endif
      for (; tau + WS_UNROLL - 1 <= t_fast1; tau += WS_UNROLL) {
#pragma unroll
        for (int u = 0; u < WS_UNROLL; u++) step(std::false_type{}, lr_tag, tau + u);
      }
#pragma unroll 1
      for (; tau < T; tau++) step(std::true_type{}, lr_tag, tau);
    };
    if (!lr_any) run(std::integral_constant<int, 0>{});
    else if (!__any_sync(FULLMASK, right || use_mail)) run(std::integral_constant<int, 1>{});
    else run(std::integral_constant<int, 2>{});
    if (A.dbg) {
      long long t_end;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
      if (lane == 0) { A.dbg[w * 4 + 0] = t_start; A.dbg[w * 4 + 1] = t_end; A.dbg[w * 4 + 2] = n_spins; }
    }
  } else if (helper) {
    /* ================================================================ helper warp */
    /* streaming: element e of a ring row <-> (layer, column) */
    const double *ld_d[Cfg::EPL_D];
    const double *ld_r[Cfg::EPL_R];
    unsigned st_d[Cfg::EPL_D], st_r[Cfg::EPL_R];
    bool ok_d[Cfg::EPL_D], ok_r[Cfg::EPL_R];
#pragma unroll
    for (int q = 0; q < Cfg::EPL_D; q++) {
      const int e = lane + 32 * q, l = e / S, xs = e % S, x = w * W + xs;
      ok_d[q] = (e < NL * S) && (x < nx || (x == nx && rint));
      ld_d[q] = A.da + (size_t)(ok_d[q] ? l : 0) * plane + GIDX(pitch, 0, ok_d[q] ? x : 0);
      st_d[q] = (unsigned)__cvta_generic_to_shared(IN) + 16u * (unsigned)((l >> 1) * S + xs) + 8u * (l & 1);
    }
#pragma unroll
    for (int q = 0; q < Cfg::EPL_R; q++) {
      const int e = lane + 32 * q, l = e / RC, xs = e % RC, x = w * W - (K - 1) + xs;
      ok_r[q] = (e < NL * RC) && (x >= 0) && (x < nx);
      ld_r[q] = A.res + (size_t)(ok_r[q] ? l : 0) * plane + GIDX(pitch, 0, ok_r[q] ? x : 0);
      st_r[q] = (unsigned)__cvta_generic_to_shared(RES) + 16u * (unsigned)((l >> 1) * RC + xs) + 8u * (l & 1);
    }
#ifndef WS_PF
#define WS_PF 48 /* rows of L2 prefetch ahead of the streamed rows */
#endif
    constexpr int PF = WS_PF;
#ifndef HROWS
    /* rows streamed in / drained per helper iteration: must outrun the compute warp.  Measured at nl = 4 (finest launch,
       us): 2: 3784, 3: 3230, 4: 3268, 5: 3256, 6: 3353 -- 3 where a row is at most as long as in the measured case */
#define HROWS (NL <= 4 ? 3 : 4)
#endif
    /* mailbox lanes: (kk, q) */
    const int kk = lane / Q, q = lane % Q;
    const bool rd_ghost = (w == 0) && lint && kk == 0; /* west column = stored halo column -1 of the iterate */
    const bool rd_valid = !MW && (rd_ghost || ((w > 0) && (wl == 0) && kk < nsw && (w * W - 1 - kk) >= 0 && (w * W - 1 - kk) < nx));
    const unsigned long long *mb_in = A.mailbox + ((size_t)(w > 0 ? w - 1 : 0) * K + kk) * (size_t)ny * NLP;
    const unsigned a_ringk = (unsigned)__cvta_generic_to_shared(XR + (size_t)kk * XRS);
    const unsigned a_ringf = (unsigned)__cvta_generic_to_shared(XR + (size_t)kf * XRS);
    const unsigned gmask = (Q == 32) ? 0xffffffffu : (((1u << Q) - 1u) << (kk * Q));
    int mail_rd = rd_valid ? 0 : ny;  /* rows deposited for sweep kk */
    int da_dr = 0;                    /* rows of the last sweep written to HBM */
    int in_issued = r_first, h1 = r_first, h2 = r_first, h3 = r_first, in_done = r_first; /* rows issued now / 1,2,3 iterations ago */
    constexpr int EPL_O = (NL * W + 31) / 32;
    int idle = 0;
    long long it = 0;
#pragma unroll 1
    for (;; it++) {
      const int cd = ld_cnt(cnt + Cfg::C_DONE);
      bool progress = false;
      /* ---- (1) mailbox in: Q rows of each sweep per iteration (the latency-critical hand-off) */
      {
        const int r = mail_rd + q;
        const bool can = rd_valid && r < ny && (cd >= r - R2 + 2 * kk + 3);
        unsigned long long v[NLP];
#pragma unroll
        for (int l = 0; l < NLP; l++) v[l] = MAIL_EMPTY;
        if (can && !rd_ghost) {
          const unsigned long long *p = mb_in + (size_t)r * NLP;
#pragma unroll
          for (int l = 0; l < NLP; l += 2)
            asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];\n" : "=l"(v[l]), "=l"(v[l + 1]) : "l"(p + l));
        }
        if (can && rd_ghost) {
#pragma unroll
          for (int l = 0; l < NL; l++) v[l] = (unsigned long long)__double_as_longlong(A.da[(size_t)l * plane + GIDX(pitch, r, -1)]);
        }
        /* ---- (2) meanwhile: stream up to HROWS rows; rows issued three iterations ago have landed */
        {
          const int rmax = min(r_last, cd + RIN - Cfg::TAIL - 2);
          const int b1 = min(in_issued + HROWS, rmax + 1);
          for (int r2 = in_issued; r2 < b1; r2++) {
            const unsigned ro = (unsigned)(r2 & (RIN - 1));
            const size_t go = (size_t)r2 * pitch;
#pragma unroll
            for (int u = 0; u < Cfg::EPL_D; u++)
              if (ok_d[u]) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(st_d[u] + ro * (DROW * 16)), "l"(ld_d[u] + go));
#pragma unroll
            for (int u = 0; u < Cfg::EPL_R; u++)
              if (ok_r[u]) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(st_r[u] + ro * (RROW * 16)), "l"(ld_r[u] + go));
            const int rp = r2 + PF;
            if (rp < ny) {
              const size_t gp = (size_t)rp * pitch;
#pragma unroll
              for (int u = 0; u < Cfg::EPL_D; u++)
                if (ok_d[u]) asm volatile("prefetch.global.L2 [%0];" ::"l"(ld_d[u] + gp));
#pragma unroll
              for (int u = 0; u < Cfg::EPL_R; u++)
                if (ok_r[u]) asm volatile("prefetch.global.L2 [%0];" ::"l"(ld_r[u] + gp));
            }
          }
          cp_async_commit();
          if (b1 > in_issued) progress = true;
          cp_async_wait<3>(); /* all but the three newest batches have landed: rows < h3 */
          h3 = h2; h2 = h1; h1 = in_issued; in_issued = b1;
        }
        /* ---- (3) last sweep's rows -> HBM, up to HROWS rows */
        {
          int done = 0;
          for (; done < HROWS; done++) {
            const int r3 = da_dr + done;
            if (!(r3 < ny && cd >= r3 + W + 2 * kf + 1)) break;
#pragma unroll
            for (int u = 0; u < EPL_O; u++) {
              const int e = lane + 32 * u, l = e / W, cs = e % W;
              const int col = w * W + cs - kf;
              if (e < NL * W && col >= 0 && col < nx) {
                double val;
                asm volatile("ld.volatile.shared.f64 %0, [%1];" : "=d"(val)
                             : "r"(a_ringf + 16u * (unsigned)((r3 & (R2 - 1)) * DROW + (l >> 1) * S + cs + 1) + 8u * (l & 1)));
                A.da[(size_t)l * plane + GIDX(pitch, r3, col)] = val;
              }
            }
          }
          da_dr += done;
          if (done > 0) progress = true;
        }
        /* ---- back to the mailbox: deposit the leading valid rows of each sweep, re-arm them */
        bool valid = can;
#pragma unroll
        for (int l = 0; l < NL; l++) valid = valid && (v[l] != MAIL_EMPTY);
        const unsigned bal = (__ballot_sync(FULLMASK, valid) & gmask) >> (kk * Q);
        const int adv = __ffs(~bal) - 1;
        if (q < adv) {
          const unsigned d = a_ringk + 16u * (unsigned)((r & (R2 - 1)) * DROW);
#pragma unroll
          for (int l = 0; l < NLP; l += 2)
            sts2(d + 16u * ((l >> 1) * S), __longlong_as_double((long long)v[l]), __longlong_as_double((long long)v[l + 1]));
          unsigned long long *p = (unsigned long long *)mb_in + (size_t)r * NLP;
          if (!rd_ghost) {
#pragma unroll
            for (int l = 0; l < NLP; l += 2)
              asm volatile("st.global.cg.v2.u64 [%0], {%1, %2};\n" ::"l"(p + l), "l"(MAIL_EMPTY), "l"(MAIL_EMPTY) : "memory");
          }
        }
        mail_rd += adv;
        if (adv > 0) progress = true;
      }
      /* ---- publish: per sweep, the last row whose inputs are complete */
      if (h3 > in_done) { in_done = h3; progress = true; }
      /* No __threadfence_block() here: it would also wait for the drain's global stores (measured: ~1 us
         per helper iteration, i.e. per hand-off).  The rings and the counters live in shared memory,
         the deposits above and the counter store below are volatile shared-memory stores of the SAME
         warp (the LSU keeps them in order), and cp.async data is complete after wait_group. */
      __syncwarp();
      if (q == 0 && kk < K) {
        int lim = (in_done > r_last) ? WS_INF : in_done - 2;
        lim = min(lim, (mail_rd >= ny) ? WS_INF : mail_rd - 1);
        if (kk == kf) lim = min(lim, (da_dr >= ny - R2) ? WS_INF : da_dr + R2 - 1);
        if (kk >= nsw) lim = WS_INF;
        cnt[(MW && wl == 0 ? Cfg::HLIM : Cfg::LIM) + kk] = lim; /* MW: the mail warp folds its own progress in */
      }
      /* ---- done? */
      const bool fin = (in_done > r_last) && (mail_rd >= ny) && (da_dr >= ny);
      if (__all_sync(FULLMASK, fin)) break;
      if (in_issued > r_last && in_done <= r_last) progress = true; /* flushing the last batches */
      if (!__any_sync(FULLMASK, progress)) {
        if (++idle > SPIN_LIMIT) { if (lane == 0) *A.err = 2; break; }
      } else idle = 0;
    }
    cp_async_wait<0>();
    if (MW && wl == 0 && lane == 0) cnt[Cfg::H_DONE] = 1;
    if (A.dbg && lane == 0) A.dbg[w * 4 + 3] = it; /* helper iterations (profiling) */
  }
  } /* w < nworkers */
}
