/*
 * rhs_kernels.cuh -- right-hand side of the PV equation and stage update.
 *
 * One RHS evaluation of the reference (update_qg, msqg/qg.h:609-650) is ~45
 * full passes over the layer lists (SURVEY.md App. C).  Here it is three:
 *   k_zeta : zeta = laplacian(psi) + dirichlet ghosts            (comp_del2, qg.h:171-181)
 *            + per-layer max|u_face|                             (comp_vel + timestep, qg.h:275-283,383-391)
 *   k_lap  : tmp  = laplacian(zeta) + ghosts                     (dissip's comp_del2, qg.h:411), only if Re/Re4 != 0
 *   k_rhs  : every tendency term in the reference's accumulation order, then
 *            the stage update q_out = q_in + dq*dt               (advance_qg, qg.h:594-606)
 * Floating-point association follows the reference expressions token by token;
 * the library is compiled with -fmad=false so results are bit-identical to an
 * x86-64 build of the reference without FMA contraction.
 */
#pragma once
#include "layout.cuh"
#include "mg_kernels.cuh"

/* laplacian macro, qg.h:169.  The reference macro has no outer parentheses, so
 * `fac*laplacian(po)` is (fac*(sum))/sq(Delta): lapf() keeps that association. */
/* Divisions by the grid constants use div_by() with host-computed reciprocals: the correctly
 * rounded IEEE quotient (same bits as `/`) in 5 fp64 ops instead of the ~30 of a generic DDIV. */
__device__ __forceinline__ double lapf(double fac, const double *__restrict__ p, size_t c, int pitch, const Geom &g) {
  return div_by(fac * (p[c + 1] + p[c - 1] + p[c + pitch] + p[c - pitch] - 4 * p[c]), g.D2, g.rD2);
}
__device__ __forceinline__ double lap5(const double *__restrict__ p, size_t c, int pitch, const Geom &g) {
  return div_by(p[c + 1] + p[c - 1] + p[c + pitch] + p[c - pitch] - 4 * p[c], g.D2, g.rD2);
}

__device__ __forceinline__ void write_ghosts(double *__restrict__ p, const Geom &g, int x, int y, double v, double sg) {
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

/* out = laplacian(in) on every layer (blockIdx.z) + dirichlet(0) ghosts.
 * If umax != NULL also reduces max |u| over the faces of layer z:
 *   u.x[i,j] = -0.25*(p[i,j+1]-p[i,j-1]+p[i-1,j+1]-p[i-1,j-1])/Delta   faces i=0..n, j=0..n-1
 *   u.y[i,j] = +0.25*(p[i+1,j]-p[i-1,j]+p[i+1,j-1]-p[i-1,j-1])/Delta   faces j=0..n, i=0..n-1
 * min over faces of Delta/|u| (timestep.h) == Delta / max|u| exactly (division
 * is monotone), so the host rebuilds the reference's dt chain from umax. */
__global__ void __launch_bounds__(256)
k_lap(const double *__restrict__ in, double *__restrict__ out, Geom g, double *__restrict__ umax, double sbcc) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  const double *p = in + (size_t)f * g.plane;
  double um = 0.;
  if (x <= g.nx && y <= g.ny) {
    const size_t c = GIDX(g.pitch, y, x);
    if (x < g.nx && y < g.ny) {
      double *o = out + (size_t)f * g.plane;
      const double v = lap5(p, c, g.pitch, g);
      o[c] = v;
      write_ghosts(o, g, x, y, v, -1.);
      if (sbcc != 0.) { /* partial slip, qg.h:185-198 */
        if (x == 0) o[c - 1] = sbcc * (p[c] - p[c - 1]);
        if (x == g.nx - 1) o[c + 1] = sbcc * (p[c] - p[c + 1]);
        if (y == 0) o[c - g.pitch] = sbcc * (p[c] - p[c - g.pitch]);
        if (y == g.ny - 1) o[c + g.pitch] = sbcc * (p[c] - p[c + g.pitch]);
      }
    }
    if (umax) {
      const int P = g.pitch;
      if (y < g.ny) { /* x-face (x, y), x = 0..nx */
        const double u = div_by(0.25 * (p[c + P] - p[c - P] + p[c - 1 + P] - p[c - 1 - P]), g.Delta, g.rD);
        const double a = fabs(u);
        if (a > um) um = a;
      }
      if (x < g.nx) { /* y-face (x, y), y = 0..ny */
        const double u = div_by(0.25 * (p[c + 1] - p[c - 1] + p[c + 1 - P] - p[c - 1 - P]), g.Delta, g.rD);
        const double a = fabs(u);
        if (a > um) um = a;
      }
    }
  }
  if (umax) block_max_to(umax + f, um);
}

/* k_lap with two cells per thread: the 3 x 4 window (rows y-1..y+1, columns x-1..x+2) is read with one 16-byte
 * and two 8-byte loads per row and serves both laplacians and all face velocities of the two cells.  The face
 * speed is reduced as max |0.25*(...)| (the numerator) and divided by Delta ONCE per block: correctly rounded
 * division is monotone and odd, so max_a |RN(x_a/Delta)| == RN(max_a |x_a| / Delta) bit for bit.
 * (ncu: the one-cell kernel above is instruction-bound at 17-29 % of DRAM peak, profiles/r01_ncu_kernels.md.)
 * Requires an even nx. */
__global__ void __launch_bounds__(256)
k_lap2(const double *__restrict__ in, double *__restrict__ out, Geom g, double *__restrict__ umax, double sbcc) {
  const int x0 = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  const double *p = in + (size_t)f * g.plane;
  double um = 0.;
  if (x0 < g.nx && y < g.ny) {
    const int P = g.pitch;
    const size_t c = GIDX(P, y, x0);
    double w[3][4]; /* w[r][k] = p(x0 - 1 + k, y - 1 + r) */
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const double *q = p + c + (ptrdiff_t)(r - 1) * P;
      const double2 m = *reinterpret_cast<const double2 *>(q);
      w[r][0] = q[-1]; w[r][1] = m.x; w[r][2] = m.y; w[r][3] = q[2];
    }
    double *o = out + (size_t)f * g.plane;
    double v[2];
#pragma unroll
    for (int k = 0; k < 2; k++) /* p[c+1] + p[c-1] + p[c+P] + p[c-P] - 4*p[c] */
      v[k] = div_by(w[1][k + 2] + w[1][k] + w[2][k + 1] + w[0][k + 1] - 4 * w[1][k + 1], g.D2, g.rD2);
    *reinterpret_cast<double2 *>(o + c) = make_double2(v[0], v[1]);
    if (x0 == 0 || x0 + 2 >= g.nx || y == 0 || y == g.ny - 1) {
      write_ghosts(o, g, x0, y, v[0], -1.);
      write_ghosts(o, g, x0 + 1, y, v[1], -1.);
      if (sbcc != 0.) { /* partial slip (sbc > 0), qg.h:185-198: zeta[ghost] = sbc/((0.5*sbc+1)*sq(Delta))*(po[]-po[ghost])
                           on the four sides, corners keep the dirichlet value */
        if (x0 == 0) o[c - 1] = sbcc * (w[1][1] - w[1][0]);
        if (x0 + 2 == g.nx) o[c + 2] = sbcc * (w[1][2] - w[1][3]);
#pragma unroll
        for (int k = 0; k < 2; k++) {
          if (y == 0) o[c + k - P] = sbcc * (w[1][k + 1] - w[0][k + 1]);
          if (y == g.ny - 1) o[c + k + P] = sbcc * (w[1][k + 1] - w[2][k + 1]);
        }
      }
    }
    if (umax) {
      double a;
#pragma unroll
      for (int k = 0; k < 2; k++) {
        /* x-face (x0+k, y): p[c+P] - p[c-P] + p[c-1+P] - p[c-1-P] */
        a = fabs(0.25 * (w[2][k + 1] - w[0][k + 1] + w[2][k] - w[0][k]));
        if (a > um) um = a;
        /* y-face (x0+k, y): p[c+1] - p[c-1] + p[c+1-P] - p[c-1-P] */
        a = fabs(0.25 * (w[1][k + 2] - w[1][k] + w[0][k + 2] - w[0][k]));
        if (a > um) um = a;
      }
      if (x0 + 2 == g.nx) { /* x-face (nx, y) */
        a = fabs(0.25 * (w[2][3] - w[0][3] + w[2][2] - w[0][2]));
        if (a > um) um = a;
      }
      if (y == g.ny - 1) { /* y-faces (x0+k, ny) */
#pragma unroll
        for (int k = 0; k < 2; k++) {
          a = fabs(0.25 * (w[2][k + 2] - w[2][k] + w[1][k + 2] - w[1][k]));
          if (a > um) um = a;
        }
      }
    }
  }
  if (umax) {
    __shared__ double sh[32];
    um = warp_max(um);
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int lane = tid & 31, wid = tid >> 5;
    const int nw = (blockDim.x * blockDim.y + 31) >> 5;
    if (lane == 0) sh[wid] = um;
    __syncthreads();
    if (wid == 0) {
      um = lane < nw ? sh[lane] : 0.;
      um = warp_max(um);
      if (lane == 0 && um > 0.) atomic_max_pos(umax + f, fabs(div_by(um, g.Delta, g.rD)));
    }
  }
}

/* jacobian macro, qg.h:252-262: returns -J(p,q), 3x3 neighbourhoods */
__device__ __forceinline__ double jac(const double *__restrict__ po, const double *__restrict__ qo, size_t c, int P,
                                      const Geom &G) {
  const long long cc = (long long)c;
#define PO(a, b) po[cc + (a) + (b) * P]
#define QO(a, b) qo[cc + (a) + (b) * P]
  return div_by(((QO(1, 0) - QO(-1, 0)) * (PO(0, 1) - PO(0, -1))
         + (QO(0, -1) - QO(0, 1)) * (PO(1, 0) - PO(-1, 0))
         + QO(1, 0) * (PO(1, 1) - PO(1, -1))
         - QO(-1, 0) * (PO(-1, 1) - PO(-1, -1))
         - QO(0, 1) * (PO(1, 1) - PO(-1, 1))
         + QO(0, -1) * (PO(1, -1) - PO(-1, -1))
         + PO(0, 1) * (QO(1, 1) - QO(-1, 1))
         - PO(0, -1) * (QO(1, -1) - QO(-1, -1))
         - PO(1, 0) * (QO(1, 1) - QO(1, -1))
         + PO(-1, 0) * (QO(-1, 1) - QO(-1, -1))),
        G.D12, G.rD12);
#undef PO
#undef QO
}

struct RhsArgs {
  const double *psi, *zeta, *tmp, *pp, *zp, *s, *qforc, *topo, *ro, *sstoch_unused;
  const double *q_in; /* stage input (advance_qg's `input`) */
  const double *q_ev; /* evolving list of this RHS (stochastic relaxation term) */
  double *q_out;      /* may alias q_in; NULL: no stage update */
  double *dq;         /* NULL: tendency not stored */
  const double *noise;     /* stochastic: n_stochl, else NULL */
  const double *wind;      /* [n] tau0/(Rom*dh0)*sin(2 pi y/L0)*sin(pi y/L0), host glibc */
  Geom g;
  double idh0[MSQG_NLMAX], idh1[MSQG_NLMAX];
  double beta, iRe, iRe4, ceks, cekb; /* ceks = Eks/(Rom*2*dh[0]), cekb = Ekb/(Rom*2*dh[nl-1]) */
  double dhb;                         /* dh[nl-1] */
  double dt, itr;
  float dts;                          /* stochastic: float, qg_stochastic.h:133-136 */
  int has_pg, has_zp, use_tmp, flag_topo, stochastic;
  int econs; /* ENERGY_CONSERV (qg.h:310-373): advect q_ev instead of zeta + J(psi_l, psi_l+1); k_rhs only */
};

/* advection_pv (qg.h:287-380; stochastic variant qg_stochastic.h:17-111),
 * dissip (:406-422), ekman_friction (:428-440), surface_forcing (:446-459),
 * qforcing (:465-474), bottom_topography (:480-488), advance_qg (:594-606;
 * stochastic qg_stochastic.h:128-149), one thread per column, layers in
 * registers so that ju = -jd is reused exactly as the reference does. */
#ifndef RHS_MINB
#define RHS_MINB 6 /* 80 registers: load latency (78 % of the stall cycles at 31 % occupancy, ncu) needs more resident warps */
#endif
template <int NL>
__global__ void __launch_bounds__(128, RHS_MINB)
k_rhs(RhsArgs A) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const Geom g = A.g;
  if (x >= g.nx || y >= g.ny) return;
  const size_t c = GIDX(g.pitch, y, x);
  const int P = g.pitch;
  const size_t pl = g.plane;
  double jd = 0., ju;
#pragma unroll
  for (int l = 0; l < NL; l++) {
    const double *po = A.psi + l * pl, *qo = A.zeta + l * pl;
    const double *pp = A.pp + l * pl;
    double dq = 0.;
    ju = -jd;
    /* --- advection_pv */
    if (l < NL - 1) {
      const double *po2 = A.psi + (l + 1) * pl, *pp2 = A.pp + (l + 1) * pl;
      if (!A.stochastic && !A.econs) {
        jd = jac(po, po2, c, P, g);
        if (A.has_pg) jd = jd + jac(pp, po2, c, P, g) + jac(po, pp2, c, P, g);
      } else { /* stochastic (qg_stochastic.h:35-36) and ENERGY_CONSERV (qg.h:311): no J(psi_l, psi_l+1) */
        jd = A.has_pg ? jac(pp, po2, c, P, g) + jac(po, pp2, c, P, g) : 0.;
      }
    }
    double adv;
    const double be = div_by(A.beta * (po[c - 1] - po[c + 1]), g.D2x, g.rD2x);
    if (!A.stochastic || l > 0) {
      adv = jac(po, A.econs ? A.q_ev + l * pl : qo, c, P, g); /* ENERGY_CONSERV: jacobian(po, qot), qg.h:312 */
      if (A.has_pg) adv = adv + jac(pp, qo, c, P, g);
      adv = adv + be;
    } else { /* stochastic top layer omits J(psi,zeta), qg_stochastic.h:39-40 */
      adv = A.has_pg ? jac(pp, qo, c, P, g) + be : be;
    }
    if (l == 0)
      adv = adv + A.s[c] * jd * A.idh1[0];
    else if (l < NL - 1)
      adv = adv + A.s[(l - 1) * pl + c] * ju * A.idh0[l] + A.s[l * pl + c] * jd * A.idh1[l];
    else
      adv = adv + A.s[(l - 1) * pl + c] * ju * A.idh0[l];
    dq += adv;
    if (A.has_zp) dq += jac(po, A.zp + l * pl, c, P, g);
    if (A.stochastic) dq += -A.q_ev[l * pl + c] * A.itr;
    /* --- dissip */
    if (A.use_tmp) {
      const double *z1 = qo, *t1 = A.tmp + l * pl;
      if (l == 0) {
        dq = 1. * dq + A.iRe * A.s[c] * (z1[pl + c] - z1[c]) * A.idh1[0];
      } else if (l < NL - 1) {
        dq = 1. * dq + A.iRe * (A.s[(l - 1) * pl + c] * (z1[c - pl] - z1[c]) * A.idh0[l] +
                                A.s[l * pl + c] * (z1[c + pl] - z1[c]) * A.idh1[l]);
      } else {
        dq = 1. * dq + A.iRe * A.s[(l - 1) * pl + c] * (z1[c - pl] - z1[c]) * A.idh0[l];
      }
      dq += t1[c] * A.iRe;
      if (l == 0) {
        dq = 1. * dq + A.iRe4 * A.s[c] * (t1[pl + c] - t1[c]) * A.idh1[0];
      } else if (l < NL - 1) {
        dq = 1. * dq + A.iRe4 * (A.s[(l - 1) * pl + c] * (t1[c - pl] - t1[c]) * A.idh0[l] +
                                 A.s[l * pl + c] * (t1[c + pl] - t1[c]) * A.idh1[l]);
      } else {
        dq = 1. * dq + A.iRe4 * A.s[(l - 1) * pl + c] * (t1[c - pl] - t1[c]) * A.idh0[l];
      }
      dq = 1. * dq + lapf(A.iRe4, t1, c, P, g);
    }
    /* --- ekman_friction */
    if (l == 0) dq -= A.ceks * qo[c];
    if (l == NL - 1) dq -= A.cekb * qo[c];
    /* --- surface_forcing */
    if (l == 0) dq -= A.wind[y];
    /* --- qforcing */
    if (A.qforc) dq += A.qforc[l * pl + c];
    /* --- bottom_topography */
    if (l == NL - 1 && A.flag_topo) dq += jac(po, A.topo, c, P, g) / (A.ro[c] * A.dhb);
    if (A.dq) A.dq[l * pl + c] = dq;
    /* --- advance_qg */
    if (A.q_out) {
      double v;
      if (!A.stochastic)
        v = A.q_in[l * pl + c] + dq * A.dt;
      else
        v = A.q_in[l * pl + c] + dq * A.dt + A.noise[l * pl + c] * A.dts;
      A.q_out[l * pl + c] = v;
    }
  }
}

/* ------------------------------------------------------------------ k_rhs_t: the same right-hand side from
 * shared-memory tiles.  k_rhs gathers ~26 doubles per cell-layer through L1 and is bound by the latency of those
 * gathers at 31-37 % occupancy (ncu: 20 % of DRAM peak, 27 % issue active).  Here a 32 x 8 block stages the
 * 34 x 10 tiles (one-cell halo; the ghost rings are stored, so the halo is always readable) of psi[l], psi[l+1],
 * zeta[l] and tmp[l] with coalesced loads -- psi[l+1] is kept for the next layer -- and the Jacobians read shared
 * memory.  Every expression is the one of k_rhs (same tokens, same association): results are bit-identical.
 * Used for the default terms (no psi_pg / zeta_pg Jacobians, no topography, not stochastic); everything else
 * stays on k_rhs. */
#define RT_X 32
#define RT_Y 8
#define RT_P (RT_X + 2) /* tile pitch */
struct TileAcc {
  const double *t; /* centre of this thread's cell in a [RT_Y+2][RT_P] shared tile */
  __device__ __forceinline__ double operator()(int a, int b) const { return t[a + b * RT_P]; }
};
template <class PA, class QA>
__device__ __forceinline__ double jac_acc(const PA PO, const QA QO, const Geom &G) {
  return div_by(((QO(1, 0) - QO(-1, 0)) * (PO(0, 1) - PO(0, -1))
         + (QO(0, -1) - QO(0, 1)) * (PO(1, 0) - PO(-1, 0))
         + QO(1, 0) * (PO(1, 1) - PO(1, -1))
         - QO(-1, 0) * (PO(-1, 1) - PO(-1, -1))
         - QO(0, 1) * (PO(1, 1) - PO(-1, 1))
         + QO(0, -1) * (PO(1, -1) - PO(-1, -1))
         + PO(0, 1) * (QO(1, 1) - QO(-1, 1))
         - PO(0, -1) * (QO(1, -1) - QO(-1, -1))
         - PO(1, 0) * (QO(1, 1) - QO(1, -1))
         + PO(-1, 0) * (QO(-1, 1) - QO(-1, -1))),
        G.D12, G.rD12);
}
/* asynchronous tile fill (LDGSTS): tile[ry*RT_P + rx] = src(y0 - 1 + ry, x0 - 1 + rx); the consumer waits with
 * cp.async.wait_group + __syncthreads, so no thread stalls on its own loads */
__device__ __forceinline__ void rt_load(double *__restrict__ tile, const double *__restrict__ src, const Geom &g, int x0, int y0, int tid) {
  constexpr int NE = (RT_Y + 2) * RT_P, NT = RT_X * RT_Y;
#pragma unroll
  for (int k = 0; k < (NE + NT - 1) / NT; k++) {
    const int e = tid + k * NT;
    const int ry = e / RT_P, rx = e - ry * RT_P;
    const int gx = x0 - 1 + rx, gy = y0 - 1 + ry;
    if (e < NE && gx <= g.nx && gy <= g.ny)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((unsigned)__cvta_generic_to_shared(tile + e)), "l"(src + GIDX(g.pitch, gy, gx)) : "memory");
  }
}
template <int NL>
__global__ void __launch_bounds__(RT_X * RT_Y)
k_rhs_t(RhsArgs A) {
  /* three tile sets in flight: layer l and l+1 are read while layer l+2 lands.  The vertical neighbours zeta[l+-1],
     tmp[l+-1] of the stretching terms come from the tile staged ahead and from a register of the layer before, so
     every plane is read once */
  constexpr int TS = (RT_Y + 2) * RT_P;
  __shared__ double sp[3][TS], sz[3][TS], st[3][TS];
  const Geom g = A.g;
  const int x0 = blockIdx.x * RT_X, y0 = blockIdx.y * RT_Y;
  const int tid = threadIdx.y * RT_X + threadIdx.x;
  const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
  const bool active = x < g.nx && y < g.ny;
  const size_t c = GIDX(g.pitch, active ? y : 0, active ? x : 0);
  const size_t pl = g.plane;
  const int tc = (threadIdx.y + 1) * RT_P + threadIdx.x + 1;
  auto stage = [&](int l) {
    if (l < NL) {
      rt_load(sp[l % 3], A.psi + l * pl, g, x0, y0, tid);
      rt_load(sz[l % 3], A.zeta + l * pl, g, x0, y0, tid);
      if (A.use_tmp) rt_load(st[l % 3], A.tmp + l * pl, g, x0, y0, tid);
    }
    cp_async_commit();
  };
  stage(0);
  stage(1);
  double jd = 0., ju;
  double zm = 0., tm = 0., sm = 0.; /* zeta, tmp, stretching of layer l-1 at this cell */
  double sl = (NL > 1) ? A.s[c] : 0., qi = (A.q_out && active) ? A.q_in[c] : 0.; /* stretching / stage input of layer l */
#pragma unroll
  for (int l = 0; l < NL; l++) {
    cp_async_wait<0>(); /* layers <= l+1 have landed (layer l+1 was issued one layer ago) */
    __syncthreads();    /* ... for every thread, and everybody is done with the buffer layer l+2 overwrites */
    stage(l + 2);
    if (active) {
      const TileAcc po{sp[l % 3] + tc}, po2{sp[(l + 1) % 3] + tc}, qo{sz[l % 3] + tc};
      const double *t1s = st[l % 3] + tc;
      /* operands of the next layer, requested before this layer's arithmetic */
      const double sn = (l + 1 < NL - 1) ? A.s[(l + 1) * pl + c] : 0.;
      const double qn = (A.q_out && l + 1 < NL) ? A.q_in[(l + 1) * pl + c] : 0.;
      double dq = 0.;
      ju = -jd;
      /* --- advection_pv */
      if (l < NL - 1) jd = jac_acc(po, po2, g);
      double adv;
      const double be = div_by(A.beta * (po(-1, 0) - po(1, 0)), g.D2x, g.rD2x);
      adv = jac_acc(po, qo, g);
      adv = adv + be;
      if (l == 0)
        adv = adv + sl * jd * A.idh1[0];
      else if (l < NL - 1)
        adv = adv + sm * ju * A.idh0[l] + sl * jd * A.idh1[l];
      else
        adv = adv + sm * ju * A.idh0[l];
      dq += adv;
      /* --- dissip */
      const double zc = qo(0, 0);
      if (A.use_tmp) {
        const double tcv = t1s[0];
        const double zp = (l < NL - 1) ? sz[(l + 1) % 3][tc] : 0., tp = (l < NL - 1) ? st[(l + 1) % 3][tc] : 0.;
        if (l == 0) {
          dq = 1. * dq + A.iRe * sl * (zp - zc) * A.idh1[0];
        } else if (l < NL - 1) {
          dq = 1. * dq + A.iRe * (sm * (zm - zc) * A.idh0[l] + sl * (zp - zc) * A.idh1[l]);
        } else {
          dq = 1. * dq + A.iRe * sm * (zm - zc) * A.idh0[l];
        }
        dq += tcv * A.iRe;
        if (l == 0) {
          dq = 1. * dq + A.iRe4 * sl * (tp - tcv) * A.idh1[0];
        } else if (l < NL - 1) {
          dq = 1. * dq + A.iRe4 * (sm * (tm - tcv) * A.idh0[l] + sl * (tp - tcv) * A.idh1[l]);
        } else {
          dq = 1. * dq + A.iRe4 * sm * (tm - tcv) * A.idh0[l];
        }
        dq = 1. * dq + div_by(A.iRe4 * (t1s[1] + t1s[-1] + t1s[RT_P] + t1s[-RT_P] - 4 * tcv), g.D2, g.rD2);
        tm = tcv;
      }
      zm = zc; sm = sl;
      /* --- ekman_friction */
      if (l == 0) dq -= A.ceks * zc;
      if (l == NL - 1) dq -= A.cekb * zc;
      /* --- surface_forcing */
      if (l == 0) dq -= A.wind[y];
      /* --- qforcing */
      if (A.qforc) dq += A.qforc[l * pl + c];
      if (A.dq) A.dq[l * pl + c] = dq;
      /* --- advance_qg */
      if (A.q_out) A.q_out[l * pl + c] = qi + dq * A.dt;
      sl = sn; qi = qn;
    }
  }
  cp_async_wait<0>();
}

/* ------------------------------------------------------------------ energy diagnostics, msqg/qg_energy.h
 * energy_tend (:228-242) in one pass: advection_de (:28-154, default build: _LS_RV, no ENERGY_CONSERV),
 * dissip_de (:157-187), ekman_friction_de (:189-204) and the running mean po_mft, every term multiplied by
 * dt*(-po*(1-ediag)+ediag) and accumulated in the reference's order.  zeta = laplacian(psi) and
 * tmp = laplacian(zeta) (with their dirichlet ghosts) are prepared by k_lap2; the two comp_stretch passes of
 * dissip_de are evaluated in place (add = 0, fac = 1: 0.*old + 1.*x == x for finite old). */
struct EnergyArgs {
  const double *psi, *zeta, *tmp, *pp, *zp, *s;
  double *de_bf, *de_vd, *de_j1, *de_j2, *de_j3, *po_mft;
  const double *qt; /* ENERGY_CONSERV: comp_q(psi) (tmp2l, qg_energy.h:33-35), else NULL */
  Geom g;
  double idh0[MSQG_NLMAX], idh1[MSQG_NLMAX];
  double beta, iRe, iRe4, ceks, cekb, dt, ediag;
  int has_pg, has_zp, nme_ft;
};

template <int NL>
__global__ void __launch_bounds__(128)
k_energy(EnergyArgs A) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const Geom g = A.g;
  if (x >= g.nx || y >= g.ny) return;
  const size_t c = GIDX(g.pitch, y, x);
  const int P = g.pitch;
  const size_t pl = g.plane;
  const double dt = A.dt, ediag = A.ediag;
  double jd_1 = 0., jd_2 = 0., jd_3 = 0., ju_1, ju_2, ju_3, jc;
#pragma unroll
  for (int l = 0; l < NL; l++) {
    const double *po = A.psi + l * pl, *qo = A.zeta + l * pl, *pp = A.pp + l * pl, *t1 = A.tmp + l * pl;
    const double w = (-po[c] * (1 - ediag) + ediag);
    ju_1 = -jd_1;
    ju_2 = -jd_3; /* swap */
    ju_3 = -jd_2; /* swap */
    if (l < NL - 1) {
      const double *po2 = A.psi + (l + 1) * pl, *pp2 = A.pp + (l + 1) * pl;
      jd_1 = jac(po, po2, c, P, g);
      jd_2 = A.has_pg ? jac(pp, po2, c, P, g) : 0.;
      jd_3 = A.has_pg ? jac(po, pp2, c, P, g) : 0.;
    }
    jc = A.has_pg ? jac(po, pp, c, P, g) : 0.;
    const double j1 = jac(po, qo, c, P, g);
    const double j2 = A.has_pg ? jac(pp, qo, c, P, g) : 0.;
    const double be = div_by(A.beta * (po[c - 1] - po[c + 1]), g.D2x, g.rD2x);
    double a1, a2, a3;
    if (l == 0) {
      const double s1 = A.s[c];
      a1 = j1 + s1 * jd_1 * A.idh1[0];
      a2 = j2 + s1 * (jd_2 + jc) * A.idh1[0];
      a3 = be + s1 * (jd_3 - jc) * A.idh1[0];
    } else if (l < NL - 1) {
      const double s0 = A.s[(l - 1) * pl + c], s1 = A.s[l * pl + c];
      a1 = j1 + s0 * ju_1 * A.idh0[l] + s1 * jd_1 * A.idh1[l];
      a2 = j2 + s0 * (ju_2 + jc) * A.idh0[l] + s1 * (jd_2 + jc) * A.idh1[l];
      a3 = be + s0 * (ju_3 - jc) * A.idh0[l] + s1 * (jd_3 - jc) * A.idh1[l];
    } else {
      const double s0 = A.s[(l - 1) * pl + c];
      a1 = j1 + s0 * ju_1 * A.idh0[l];
      a2 = j2 + s0 * (ju_2 + jc) * A.idh0[l];
      a3 = be + s0 * (ju_3 - jc) * A.idh0[l];
    }
    if (A.qt) a1 = jac(po, A.qt + l * pl, c, P, g); /* ENERGY_CONSERV, qg_energy.h:66,102,134 */
    A.de_j1[l * pl + c] += a1 * dt * w;
    if (A.has_pg) A.de_j2[l * pl + c] += a2 * dt * w;
    double d3 = A.de_j3[l * pl + c];
    d3 += a3 * dt * w;
    if (A.has_zp) d3 += jac(po, A.zp + l * pl, c, P, g) * dt * w;
    A.de_j3[l * pl + c] = d3;
    /* dissip_de */
    if (A.iRe != 0. || A.iRe4 != 0.) {
      double str, str2;
      if (l == 0) {
        str = 1. * A.s[c] * (qo[pl + c] - qo[c]) * A.idh1[0];
        str2 = 1. * A.s[c] * (t1[pl + c] - t1[c]) * A.idh1[0];
      } else if (l < NL - 1) {
        str = 1. * (A.s[(l - 1) * pl + c] * (qo[c - pl] - qo[c]) * A.idh0[l] + A.s[l * pl + c] * (qo[c + pl] - qo[c]) * A.idh1[l]);
        str2 = 1. * (A.s[(l - 1) * pl + c] * (t1[c - pl] - t1[c]) * A.idh0[l] + A.s[l * pl + c] * (t1[c + pl] - t1[c]) * A.idh1[l]);
      } else {
        str = 1. * A.s[(l - 1) * pl + c] * (qo[c - pl] - qo[c]) * A.idh0[l];
        str2 = 1. * A.s[(l - 1) * pl + c] * (t1[c - pl] - t1[c]) * A.idh0[l];
      }
      double dv = A.de_vd[l * pl + c];
      dv += (t1[c] + str) * A.iRe * dt * w;
      dv += lapf(A.iRe4, t1, c, P, g) * dt * w;
      dv += A.iRe4 * (str2) * dt * w;
      A.de_vd[l * pl + c] = dv;
    }
    /* ekman_friction_de */
    if (l == 0) A.de_bf[c] -= A.ceks * qo[c] * dt * w;
    if (l == NL - 1) A.de_bf[l * pl + c] -= A.cekb * qo[c] * dt * w;
    /* running mean of psi for filter_de */
    A.po_mft[l * pl + c] = (A.po_mft[l * pl + c] * A.nme_ft + po[c]) / (A.nme_ft + 1);
  }
}

/* ------------------------------------------------------------------ passive tracers
 * ptr_rhs (msqg/qg.h:573-588): dpdt += jacobian(po, ptr) + iPe*laplacian(ptr) + ptr_ir*(ptr_relax - ptr) with
 * dpdt zeroed before (:611-613), fused with the stage update ptr_out = ptr_in + dpdt*dt (advance_qg, :597-603)
 * and the zero-gradient boundary of the tracer lists (create_layer_var(.., bc_type+1), :868).  One thread per
 * cell, blockIdx.z = scalar index f = l*nptr + nt. */
struct PtrArgs {
  const double *psi, *ptr, *relax, *ptr_in;
  double *ptr_out, *dptr;
  Geom g;
  double iPe[MSQG_MAXL], ptr_ir[MSQG_MAXL];
  double dt;
  int nptr;
};
__global__ void __launch_bounds__(256)
k_ptr_rhs(PtrArgs A) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  const Geom g = A.g;
  if (x >= g.nx || y >= g.ny) return;
  const int l = f / A.nptr, nt = f % A.nptr;
  const size_t c = GIDX(g.pitch, y, x), pl = g.plane;
  const double *po = A.psi + l * pl, *tr = A.ptr + f * pl;
  double dp = 0.;
  dp += jac(po, tr, c, g.pitch, g) + lapf(A.iPe[nt], tr, c, g.pitch, g) + A.ptr_ir[nt] * (A.relax[f * pl + c] - tr[c]);
  if (A.dptr) A.dptr[f * pl + c] = dp;
  if (A.ptr_out) {
    const double v = A.ptr_in[f * pl + c] + dp * A.dt;
    A.ptr_out[f * pl + c] = v;
    write_ghosts(A.ptr_out + f * pl, g, x, y, v, 1.);
  }
}

/* advance_qg alone (API parity with the function-pointer plugin, qg.h:594-606) */
__global__ void k_advance(double *__restrict__ out, const double *__restrict__ in, const double *__restrict__ dq,
                          const double *__restrict__ noise, Geom g, double dt, float dts) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int f = blockIdx.z;
  if (x >= g.nx || y >= g.ny) return;
  const size_t c = (size_t)f * g.plane + GIDX(g.pitch, y, x);
  if (noise)
    out[c] = in[c] + dq[c] * dt + noise[c] * dts;
  else
    out[c] = in[c] + dq[c] * dt;
}

/* comp_q: q = laplacian(psi) + stretching(psi)  (qg.h:396-403 -> :171-181, :202-246) */
template <int NL>
__global__ void __launch_bounds__(256)
k_comp_q(const double *__restrict__ psi, const double *__restrict__ s, double *__restrict__ q, Geom g, LayerMetrics M) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= g.nx || y >= g.ny) return;
  const size_t c = GIDX(g.pitch, y, x);
  const size_t pl = g.plane;
#pragma unroll
  for (int l = 0; l < NL; l++) {
    const double *p = psi + l * pl;
    double v = 0. * 0. + 1. * lap5(p, c, g.pitch, g);
    if (l == 0)
      v = 1. * v + 1. * s[c] * (p[pl + c] - p[c]) * M.idh1[0];
    else if (l < NL - 1)
      v = 1. * v + 1. * (s[(l - 1) * pl + c] * (p[c - pl] - p[c]) * M.idh0[l] + s[l * pl + c] * (p[c + pl] - p[c]) * M.idh1[l]);
    else
      v = 1. * v + 1. * s[(l - 1) * pl + c] * (p[c - pl] - p[c]) * M.idh0[l];
    q[l * pl + c] = v;
    write_ghosts(q + l * pl, g, x, y, v, -1.);
  }
}

/* modal projections, invertq's MODE_PV_INVERT branch (qg.h:118-131, :144-157):
 *   out_m = sum_l mat[m*nl+l] * in_l   accumulated from 0. in the reference order.
 * The matrices are fields in the reference (nl^2 scalars per column); they are
 * kept as fields here only when they vary in space, else passed as constants. */
template <int NL>
struct ModeMat {
  double a[NL * NL];
};

/* RING (tiles): the threads cover the interior plus the one-cell ring, and project the ring cells of the INTERNAL sides
 * too (cells of a neighbouring tile whose input holds the owner's bits, so the output does as well); the ghosts of the
 * physical sides are left to k_ghosts, and `ghosts` is ignored */
template <int NL, bool RING = false>
__global__ void __launch_bounds__(256)
k_project(const double *__restrict__ in, double *__restrict__ out, Geom g, ModeMat<NL> M,
          const double *__restrict__ matf /* optional per-cell matrix planes */, int ghosts) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x - (RING ? 1 : 0);
  const int y = blockIdx.y * blockDim.y + threadIdx.y - (RING ? 1 : 0);
  if (RING) {
    if (x > g.nx || y > g.ny) return;
    const bool okx = x < 0 ? (g.bc & 1) : (x >= g.nx ? (g.bc & 2) : true);
    const bool oky = y < 0 ? (g.bc & 4) : (y >= g.ny ? (g.bc & 8) : true);
    if (!okx || !oky) return;
    ghosts = 0;
  } else if (x >= g.nx || y >= g.ny)
    return;
  const size_t c = GIDX(g.pitch, y, x);
  const size_t pl = g.plane;
  double v[NL];
#pragma unroll
  for (int l = 0; l < NL; l++) v[l] = in[l * pl + c];
#pragma unroll
  for (int m = 0; m < NL; m++) {
    double acc = 0.;
#pragma unroll
    for (int l = 0; l < NL; l++) acc += (matf ? matf[(size_t)(m * NL + l) * pl + c] : M.a[m * NL + l]) * v[l];
    out[m * pl + c] = acc;
    if (ghosts) write_ghosts(out + m * pl, g, x, y, acc, -1.);
  }
}

/* ke_1 of writestdout (qg.c:101-106): ke -= 0.5*psi0*laplacian(psi0)*sq(Delta).
 * The reference sums in traversal order; a parallel sum differs in the last
 * bits, so this is a diagnostic (deterministic two-stage tree), not a parity
 * quantity. */
__global__ void __launch_bounds__(256)
k_ke_partial(const double *__restrict__ p, Geom g, double *__restrict__ part) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  double v = 0.;
  if (x < g.nx && y < g.ny) {
    const size_t c = GIDX(g.pitch, y, x);
    v = lapf(0.5 * p[c], p, c, g.pitch, g) * (g.Delta * g.Delta);
  }
  __shared__ double sh[256];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  sh[tid] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) sh[tid] += sh[tid + o];
    __syncthreads();
  }
  if (tid == 0) part[blockIdx.y * gridDim.x + blockIdx.x] = sh[0];
}


/* ------------------------------------------------------------------ stochastic forcing, production noise mode
 * The reference draws n = amp * sigma * N(0,1) with Box-Muller on sequential libc rand() (qg_stochastic.h:9,117-126);
 * that stream is replayed on the host in the parity mode.  Here the same transform runs on a counter-based generator
 * (Philox4x32-10, counter = (cell-layer index, draw number), key = (seed, tag)), so a field of noise is one kernel and
 * does not depend on traversal order or on how many members share a GPU.  oracle/msqg_oracle.c mirrors it.
 * The counter is the GLOBAL cell-layer index (l*N + y0 + y)*N + x0 + x, with (x0, y0) the origin of the tile in the
 * n x n grid: a decomposed or periodic group draws, cell by cell, the bits of the undecomposed field (where x0 = y0 = 0
 * and n = g.nx = g.ny, the index of the whole grid). */
__device__ __forceinline__ void philox4x32_10(unsigned int (&c)[4], unsigned int k0, unsigned int k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned int hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const unsigned int hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const unsigned int n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
__global__ void __launch_bounds__(256)
k_noise_philox(double *__restrict__ noise, const double *__restrict__ sigma, Geom g, int n, int x0, int y0, double amp,
               unsigned int seed, unsigned long long draw) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int l = blockIdx.z;
  if (x >= g.nx || y >= g.ny) return;
  const unsigned long long idx = ((unsigned long long)l * n + y0 + y) * n + x0 + x;
  unsigned int c[4] = {(unsigned int)idx, (unsigned int)(idx >> 32), (unsigned int)draw, (unsigned int)(draw >> 32)};
  philox4x32_10(c, seed, 0x6d737167u);
  const double u1 = (((double)c[0]) * 4294967296. + (double)c[1] + 0.5) * (1. / 18446744073709551616.);
  const double u2 = (((double)c[2]) * 4294967296. + (double)c[3] + 0.5) * (1. / 18446744073709551616.);
  const double gsn = sqrt(-2. * log(u1)) * cos(2 * 3.14159265358979323846 * u2);
  const size_t cc = (size_t)l * g.plane + GIDX(g.pitch, y, x);
  const double v = amp * sigma[cc] * gsn;
  double *p = noise + (size_t)l * g.plane;
  p[GIDX(g.pitch, y, x)] = v;
  /* the ghosts of the reference's boundary(n_stochl); nothing reads them (the stochastic terms of k_rhs and k_advance
     are pointwise), so on a tile the ring is left as written here and never exchanged with the neighbours */
  write_ghosts(p, g, x, y, v, -1.);
}
