/*
 * msqg_oracle.c -- CPU oracle (TEST INFRASTRUCTURE ONLY, see msqg_oracle.h).
 *
 * Plain C99 restatement of the reference msqg timestep.  Loop nests follow the
 * reference traversal order (Basilisk multigrid foreach(): x outer, y inner,
 * layer loops innermost as written in the source), which *is* the
 * Gauss-Seidel order of relax_layer.  Floating-point association follows the
 * reference expressions token by token; build with -ffp-contract=off.
 *
 * PARITY UNPINNED (no reference golden vectors exist; see header).
 *
 * Citations "qg.h:NNN" etc. are relative to /root/reference/msqg/ unless a
 * directory is given.  "[BASILISK]" marks behaviour of the Basilisk runtime
 * (not in the reference tree) restated from its published source; the in-tree
 * corroborating copy is cited where one exists.
 */
#define _GNU_SOURCE
#include "msqg_oracle.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <sys/types.h>

#define sq(x) ((x) * (x))
#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#define pi M_PI
#define HUGEV 1e30
#define TEPS 1e-9

enum { BC_DIRICHLET0 = 0, BC_NEUMANN = 1, BC_PERIODIC = 2 };

/* ------------------------------------------------------------------ grid
 * [BASILISK] grid/multigrid.h: levels 0..depth, level l has 2^l x 2^l cells,
 * Delta_l = L0/2^l, one ghost ring is all msqg ever reads.
 * Storage here: per scalar per level, (n+2)^2 doubles, y fastest. */
typedef struct {
  int nf, bc, depth;
  double **d; /* d[f*(depth+1)+l] */
} flist;

static inline int LN(int l) { return 1 << l; }
#define IDX(n, i, j) (((size_t)((i) + 1)) * (size_t)((n) + 2) + (size_t)((j) + 1))

static flist fl_new(int nf, int bc, int depth) {
  flist f;
  f.nf = nf; f.bc = bc; f.depth = depth;
  f.d = (double **)calloc((size_t)nf * (depth + 1), sizeof(double *));
  for (int k = 0; k < nf; k++)
    for (int l = 0; l <= depth; l++) {
      size_t n = LN(l);
      f.d[k * (depth + 1) + l] = (double *)calloc((n + 2) * (n + 2), sizeof(double));
    }
  return f;
}
static void fl_free(flist *f) {
  if (!f->d) return;
  for (int k = 0; k < f->nf * (f->depth + 1); k++) free(f->d[k]);
  free(f->d); f->d = NULL;
}
static inline double *FL(const flist *f, int k, int l) { return f->d[k * (f->depth + 1) + l]; }
static void fl_copy_level(flist *dst, const flist *src, int l) {
  size_t n = LN(l);
  for (int k = 0; k < src->nf; k++)
    memcpy(FL(dst, k, l), FL(src, k, l), (n + 2) * (n + 2) * sizeof(double));
}

/* [BASILISK] box_boundary_level (grid/cartesian-common / multigrid): sides in
 * the order right, left, top, bottom; each side's loop runs over the full
 * tangential range *including ghosts*, so corners end up with the y-BC applied
 * to the x-ghost.  dirichlet(0): ghost = -interior (layer.h:17-21);
 * default (symmetry): ghost = interior.
 * periodic(right); periodic(top) (qg.h:842-846, sbc = -1): the ghost ring holds the cells of the opposite side,
 * the y pass again runs over the x ghosts, so a corner holds the diagonally opposite cell; like every ghost it is
 * only refreshed by boundary calls (a Gauss-Seidel sweep reads the pre-sweep value across the seam). */
static void boundary_level(flist *f, int l) {
  int n = LN(l);
  double sg = (f->bc == BC_DIRICHLET0) ? -1. : 1.;
  for (int k = 0; k < f->nf; k++) {
    double *a = FL(f, k, l);
    if (f->bc == BC_PERIODIC) {
      for (int j = -1; j <= n; j++) a[IDX(n, n, j)] = a[IDX(n, 0, j)];
      for (int j = -1; j <= n; j++) a[IDX(n, -1, j)] = a[IDX(n, n - 1, j)];
      for (int i = -1; i <= n; i++) a[IDX(n, i, n)] = a[IDX(n, i, 0)];
      for (int i = -1; i <= n; i++) a[IDX(n, i, -1)] = a[IDX(n, i, n - 1)];
      continue;
    }
    for (int j = -1; j <= n; j++) a[IDX(n, n, j)] = sg * a[IDX(n, n - 1, j)]; /* right */
    for (int j = -1; j <= n; j++) a[IDX(n, -1, j)] = sg * a[IDX(n, 0, j)];    /* left */
    for (int i = -1; i <= n; i++) a[IDX(n, i, n)] = sg * a[IDX(n, i, n - 1)]; /* top */
    for (int i = -1; i <= n; i++) a[IDX(n, i, -1)] = sg * a[IDX(n, i, 0)];    /* bottom */
  }
}
static void boundary(flist *f) { boundary_level(f, f->depth); }

/* [BASILISK] restriction(): for l = depth-1..0, coarse = average of the 4
 * children (restriction_average: sum over foreach_child() in the order
 * (0,0),(0,1),(1,0),(1,1), x outer; then /4), then boundary_level(l). */
static void restriction(flist *f) {
  for (int l = f->depth - 1; l >= 0; l--) {
    int n = LN(l), nf2 = 2 * n;
    for (int k = 0; k < f->nf; k++) {
      double *c = FL(f, k, l);
      const double *a = FL(f, k, l + 1);
#pragma omp parallel for schedule(static)
      for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
          double sum = 0.;
          sum += a[IDX(nf2, 2 * i, 2 * j)];
          sum += a[IDX(nf2, 2 * i, 2 * j + 1)];
          sum += a[IDX(nf2, 2 * i + 1, 2 * j)];
          sum += a[IDX(nf2, 2 * i + 1, 2 * j + 1)];
          c[IDX(n, i, j)] = sum / 4;
        }
    }
    boundary_level(f, l);
  }
}

/* [BASILISK] bilinear(point,s), 2-D:
 * (9*coarse(s) + 3*(coarse(s,child.x) + coarse(s,0,child.y)) + coarse(s,child.x,child.y))/16 */
static void prolong_level(flist *f, int l) {
  int n = LN(l), nc = n / 2;
  for (int k = 0; k < f->nf; k++) {
    double *a = FL(f, k, l);
    const double *c = FL(f, k, l - 1);
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        int ic = i >> 1, jc = j >> 1;
        int cx = (i & 1) ? 1 : -1, cy = (j & 1) ? 1 : -1;
        a[IDX(n, i, j)] = (9. * c[IDX(nc, ic, jc)] +
                           3. * (c[IDX(nc, ic + cx, jc)] + c[IDX(nc, ic, jc + cy)]) +
                           c[IDX(nc, ic + cx, jc + cy)]) / 16.;
      }
  }
}

/* ------------------------------------------------------------------ model */
struct orc_model {
  orc_params p;
  int N, nl, depth;
  double L0;
  /* qg.h:7-10 */
  double *dhf, *dhc, *idh0, *idh1;
  /* qg.h:23-59 */
  flist pol, qol, zetal, zetapl, q_forcl, tmpl, ppl, Frl, strl;
  flist qom, pom, iBul, cl2m, cm2l;
  flist Ro, Rd, topo, sig_filt;
  flist sig_lev, qofl, wvl; /* qg.h:49 (all levels), qg.h:27 filter mean, scratch wavelet coefficients */
  int nbar;                 /* qg.h:86 */
  flist dql;    /* "updates" */
  flist qpred;  /* "predictor" */
  flist s_stochl, n_stochl;
  /* qg_energy.h:7-17 */
  flist de_bfl, de_vdl, de_j1l, de_j2l, de_j3l, de_ftl, tmp2l, po_mft;
  /* passive tracers, qg.h:100-101,867-870 (+ their predictor and updates: the tail of [BASILISK]'s evolving lists) */
  flist ptracersl, ptr_relaxl, ptr_pred, dptrl;
  int nme_ft, energy_vars;
  int flag_topo;
  double iRe, iRe4, Eks, Ekb;
  /* timestep() static, [BASILISK] timestep.h; copy newqg/qg.h:202-219 */
  double ts_previous;
  int corrector_step; /* qg_stochastic.h:3 */
  double t; int iter; double dt;
  orc_mgstats mgpsi, mgmode[ORC_MAXL];
  int total_cycles;
  int agg_n; /* MPI-emulation: levels with n < agg_n are swept as one block */
  int noise_mode; unsigned int noise_seed; unsigned long long noise_draw; /* orc_set_noise_mode */
  int energy_conserv; /* the reference's -DENERGY_CONSERV=1 build (qg.h:310-373, qg_energy.h:33-140) as a runtime switch */
  int smoother; /* 0: the reference's lexicographic sweep; 1: red-black ordering of the same cell update (orc_set_smoother) */
};

/* create_layer_var, layer.h:5-35 */
static flist create_layer_var(int nf, int bc_type, int depth) {
  /* bc_type 0: dirichlet(0) on the four sides; > 0: [BASILISK]'s default (symmetry); < 0: nothing set after
     periodic(right), periodic(top) (qg.h:842-846: bc_type = -2, and bc_type + 1 = -1 for Frl / strl) */
  flist f = fl_new(nf, bc_type == 0 ? BC_DIRICHLET0 : (bc_type < 0 ? BC_PERIODIC : BC_NEUMANN), depth);
  boundary(&f);
  return f;
}

void orc_default_params(orc_params *p) {
  memset(p, 0, sizeof(*p));
  /* [BASILISK] defaults N=64, L0=1, DT=1e10, CFL=0.5 ; qg.h:53-98 */
  p->N = 64; p->nl = 1; p->ediag = -1; p->L0 = 1.; p->beta = 0.5;
  p->afilt = 10.; p->Lfmax = 1.e10; p->DT = 1e10; p->tend = 1; p->dtout = 1;
  p->dtflt = -1; p->CFL = 0.5; p->amp_stoch = 1; p->px = p->py = 1;
}

/* trim_whitespace, qg.h:668-675: strips blanks only */
static void trim_ws(char *s) {
  const char *d = s;
  do { while (*d == ' ') ++d; } while ((*s++ = *d++));
}
/* str2array, qg.h:678-687 */
static void str2array(char *s, double *arr) {
  int n = 0;
  char *p = strtok(s, "[,]");
  while (p != NULL && n < ORC_MAXL) { arr[n++] = atof(p); p = strtok(NULL, ","); }
}
static void derive_params(orc_params *p) {
  /* qg.h:739-746 */
  if (p->Re == 0) p->iRe = 0.; else p->iRe = 1 / p->Re;
  if (p->Re4 == 0) p->iRe4 = 0.; else p->iRe4 = -1 / p->Re4;
  if (p->Re != 0) p->DT = 0.5 * fmin(p->DT, sq(p->L0 / p->N) * p->Re / 4.);
  if (p->Re4 != 0) p->DT = 0.5 * fmin(p->DT, sq(sq(p->L0 / p->N)) * p->Re4 / 32.);
  if (p->tr_stoch != 0) p->itr_stoch = 1 / p->tr_stoch; /* qg.h:757 */
  for (int nt = 0; nt < p->nptr && nt < ORC_MAXL; nt++) { /* qg.h:751-754 */
    if (p->ptr_r[nt] == 0) p->ptr_ir[nt] = 0.; else p->ptr_ir[nt] = 1 / p->ptr_r[nt];
    if (p->Pe[nt] == 0) p->iPe[nt] = 0.; else p->iPe[nt] = 1 / p->Pe[nt];
  }
}
int orc_read_params(const char *path, orc_params *p) {
  FILE *fp = fopen(path, "rt");
  if (!fp) return -1;
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
    else if (!strcmp(k, "tr_stoch"))  p->tr_stoch = atof(v);
    else if (!strcmp(k, "amp_stoch")) p->amp_stoch = atof(v);
  }
  fclose(fp);
  derive_params(p);
  return 0;
}

/* set_vars, qg.h:837-925 (+ set_vars_stoch, qg_stochastic.h:153-172) */
orc_model *orc_create(const orc_params *p) {
  orc_model *m = (orc_model *)calloc(1, sizeof(orc_model));
  m->p = *p;
  m->N = p->N; m->nl = p->nl; m->L0 = p->L0;
  int depth = 0;
  while ((1 << depth) < p->N) depth++;
  m->depth = depth;
  int nl = p->nl, bc = 0;
  if (p->sbc == -1) bc = -2; /* qg.h:842-846 */
  const int bcs = bc < 0 ? -1 : 1; /* plain `scalar x[]` globals: default boundaries, periodic after periodic() */
  m->pol = create_layer_var(nl, bc, depth);
  m->qol = create_layer_var(nl, bc, depth);
  m->ppl = create_layer_var(nl, bc, depth);
  m->zetal = create_layer_var(nl, bc, depth);
  m->zetapl = create_layer_var(nl, bc, depth);
  m->q_forcl = create_layer_var(nl, bc, depth);
  m->tmpl = create_layer_var(nl, bc, depth);
  m->Frl = create_layer_var(nl, bc + 1, depth);
  m->strl = create_layer_var(nl, bc + 1, depth);
  m->dql = create_layer_var(nl, bc, depth);
  m->qpred = create_layer_var(nl, bc, depth);
  if (p->mode_pv_invert) {
    m->pom = create_layer_var(nl, bc, depth);
    m->qom = create_layer_var(nl, bc, depth);
    m->iBul = create_layer_var(nl, bc + 1, depth);
    m->cl2m = create_layer_var(nl * nl, bc + 1, depth);
    m->cm2l = create_layer_var(nl * nl, bc + 1, depth);
  }
  if (p->stochastic) {
    m->s_stochl = create_layer_var(nl, 0, depth); /* qg_stochastic.h:157-159: bc_type = 0 whatever sbc is */
    m->n_stochl = create_layer_var(nl, 0, depth);
  }
  if (p->nptr > 0) { /* qg.h:867-870: bc_type+1 (Basilisk's default, zero-gradient, boundaries); clones inherit them */
    m->ptracersl = create_layer_var(nl * p->nptr, bc + 1, depth);
    m->ptr_relaxl = create_layer_var(nl * p->nptr, bc + 1, depth);
    m->ptr_pred = create_layer_var(nl * p->nptr, bc + 1, depth);
    m->dptrl = create_layer_var(nl * p->nptr, bc + 1, depth);
  }
  m->Ro = create_layer_var(1, bcs, depth);
  m->Rd = create_layer_var(1, bcs, depth);
  m->topo = create_layer_var(1, bcs, depth);
  m->sig_filt = create_layer_var(1, bcs, depth);
  m->sig_lev = create_layer_var(1, bcs, depth);
  m->qofl = create_layer_var(nl, bc, depth);   /* qg.h:860 */
  m->wvl = create_layer_var(1, 0, depth);      /* scalar w[] with w[top] = w[bottom] = w[right] = w[left] = 0, qg.h:525-529 */
  m->dhc = (double *)calloc(nl, sizeof(double));
  m->dhf = (double *)calloc(nl, sizeof(double));
  m->idh0 = (double *)calloc(nl, sizeof(double));
  m->idh1 = (double *)calloc(nl, sizeof(double));
  for (int l = 0; l < nl; l++) m->dhf[l] = p->dh[l];
  int n = m->N;
  double Delta = m->L0 / n;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double x = (i + 0.5) * Delta, y = (j + 0.5) * Delta;
      for (int l = 0; l < nl - 1; l++) FL(&m->Frl, l, depth)[IDX(n, i, j)] = p->Fr[l];
      for (int l = 0; l < nl; l++)
        FL(&m->ppl, l, depth)[IDX(n, i, j)] = p->vpg[l] * x - p->upg[l] * y;
      FL(&m->Ro, 0, depth)[IDX(n, i, j)] = p->Rom;
      FL(&m->Rd, 0, depth)[IDX(n, i, j)] = 1.;
      FL(&m->topo, 0, depth)[IDX(n, i, j)] = 0.;
    }
  boundary(&m->ppl);
  m->iRe = p->iRe; m->iRe4 = p->iRe4; m->Eks = p->Eks; m->Ekb = p->Ekb;
  m->ts_previous = 0.;
  m->agg_n = 0;
  return m;
}

void orc_destroy(orc_model *m) {
  if (!m) return;
  flist *all[] = {&m->pol, &m->qol, &m->zetal, &m->zetapl, &m->q_forcl, &m->tmpl, &m->ppl,
                  &m->Frl, &m->strl, &m->qom, &m->pom, &m->iBul, &m->cl2m, &m->cm2l, &m->Ro,
                  &m->Rd, &m->topo, &m->sig_filt, &m->sig_lev, &m->qofl, &m->wvl, &m->dql, &m->qpred, &m->s_stochl, &m->n_stochl,
                  &m->de_bfl, &m->de_vdl, &m->de_j1l, &m->de_j2l, &m->de_j3l, &m->de_ftl, &m->tmp2l, &m->po_mft,
                  &m->ptracersl, &m->ptr_relaxl, &m->ptr_pred, &m->dptrl};
  for (size_t k = 0; k < sizeof(all) / sizeof(all[0]); k++) fl_free(all[k]);
  free(m->dhc); free(m->dhf); free(m->idh0); free(m->idh1);
  free(m);
}

static flist *list_by_id(orc_model *m, int id) {
  switch (id) {
    case ORC_PSI: return &m->pol;   case ORC_Q: return &m->qol;
    case ORC_PSIPG: return &m->ppl; case ORC_FR: return &m->Frl;
    case ORC_QFORC: return &m->q_forcl; case ORC_TOPO: return &m->topo;
    case ORC_RD: return &m->Rd;     case ORC_SSTOCH: return &m->s_stochl;
    case ORC_ZETA: return &m->zetal; case ORC_DQ: return &m->dql;
    case ORC_STR: return &m->strl;  case ORC_NSTOCH: return &m->n_stochl;
    case ORC_IBU: return &m->iBul;  case ORC_CL2M: return &m->cl2m;
    case ORC_CM2L: return &m->cm2l; case ORC_PM: return &m->pom;
    case ORC_QM: return &m->qom;    case ORC_TMP: return &m->tmpl;
    case ORC_ZETAP: return &m->zetapl;
    case ORC_DE_BF: return &m->de_bfl; case ORC_DE_VD: return &m->de_vdl;
    case ORC_DE_J1: return &m->de_j1l; case ORC_DE_J2: return &m->de_j2l;
    case ORC_DE_J3: return &m->de_j3l; case ORC_DE_FT: return &m->de_ftl;
    case ORC_PO_MFT: return &m->po_mft;
    case ORC_PTR: return &m->ptracersl; case ORC_PTR_RELAX: return &m->ptr_relaxl;
    case ORC_DPTR: return &m->dptrl;
    case ORC_QOF: return &m->qofl; case ORC_SIGLEV: return &m->sig_lev;
  }
  return NULL;
}
int orc_nfields(orc_model *m, int id) { flist *f = list_by_id(m, id); return f && f->d ? f->nf : 0; }

/* pyset_field / pyget_field, qg.h:1164-1189: numpy [l][y][x] <-> cells */
static void set_list(flist *f, int N, const double *v) {
  int D = f->depth;
  for (int k = 0; k < f->nf; k++)
    for (int i = 0; i < N; i++)
      for (int j = 0; j < N; j++)
        FL(f, k, D)[IDX(N, i, j)] = v[(size_t)N * N * k + (size_t)N * j + i];
  boundary(f);
}
static void get_list(const flist *f, int N, double *v) {
  int D = f->depth;
  for (int k = 0; k < f->nf; k++)
    for (int i = 0; i < N; i++)
      for (int j = 0; j < N; j++)
        v[(size_t)N * N * k + (size_t)N * j + i] = FL(f, k, D)[IDX(N, i, j)];
}
void orc_set_field(orc_model *m, int id, const double *v) {
  flist *f = list_by_id(m, id);
  if (f && f->d) set_list(f, m->N, v);
}
void orc_get_field(orc_model *m, int id, double *v) {
  flist *f = list_by_id(m, id);
  if (f && f->d) get_list(f, m->N, v);
}
void orc_set_flag_topo(orc_model *m, int flag) { m->flag_topo = flag; }
void orc_set_decomp(orc_model *m, int px, int py, int agg_n) { m->p.px = px; m->p.py = py; m->agg_n = agg_n; }
void orc_set_noise_mode(orc_model *m, int mode, unsigned seed) { m->noise_mode = mode == 1; m->noise_seed = seed; m->noise_draw = 0; }
void orc_set_smoother(orc_model *m, int smoother) { m->smoother = smoother == 1 ? 1 : 0; }
int orc_get_smoother(orc_model *m) { return m->smoother; }
/* the reference's compile-time variant -DENERGY_CONSERV=1 (qg.h:310-373, qg_energy.h:33-140) as a runtime switch */
void orc_set_energy_conserv(orc_model *m, int on) { m->energy_conserv = on ? 1 : 0; }

/* ------------------------------------------------------------ operators */
/* laplacian macro, qg.h:169.  Like the reference's it has NO outer parentheses:
 * `fac*laplacian(po)` therefore associates as (fac*(sum))/sq(Delta), and the
 * ke_1 expression of qg.c:106 as ((0.5*po*(sum))/sq(Delta))*sq(Delta). */
#define LAP(a, n, i, j, D)                                                            \
  (a[IDX(n, (i) + 1, j)] + a[IDX(n, (i) - 1, j)] + a[IDX(n, i, (j) + 1)] +            \
   a[IDX(n, i, (j) - 1)] - 4 * a[IDX(n, i, j)]) / (sq(D))

/* comp_del2, qg.h:171-200 (sbc >= 0; the periodic variant sbc = -1 is out of scope) */
static void comp_del2(orc_model *m, flist *pl, flist *zl, double add, double fac) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n;
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        const double *po = FL(pl, l, D);
        double *ze = FL(zl, l, D);
        ze[IDX(n, i, j)] = add * ze[IDX(n, i, j)] + fac * LAP(po, n, i, j, Delta);
      }
  boundary(zl);
  /* partial slip, qg.h:185-198: the vorticity ghosts on the four sides (not the corners) */
  double sbc = m->p.sbc;
  if (sbc > 0) {
    for (int l = 0; l < nl; l++) {
      const double *po = FL(pl, l, D);
      double *ze = FL(zl, l, D);
      for (int j = 0; j < n; j++) ze[IDX(n, -1, j)] = sbc / ((0.5 * sbc + 1) * sq(Delta)) * (po[IDX(n, 0, j)] - po[IDX(n, -1, j)]);
      for (int j = 0; j < n; j++) ze[IDX(n, n, j)] = sbc / ((0.5 * sbc + 1) * sq(Delta)) * (po[IDX(n, n - 1, j)] - po[IDX(n, n, j)]);
      for (int i = 0; i < n; i++) ze[IDX(n, i, n)] = sbc / ((0.5 * sbc + 1) * sq(Delta)) * (po[IDX(n, i, n - 1)] - po[IDX(n, i, n)]);
      for (int i = 0; i < n; i++) ze[IDX(n, i, -1)] = sbc / ((0.5 * sbc + 1) * sq(Delta)) * (po[IDX(n, i, 0)] - po[IDX(n, i, -1)]);
    }
  }
}

/* comp_stretch, qg.h:202-246 */
static void comp_stretch(orc_model *m, flist *pl, flist *sl, double add, double fac) {
  int n = m->N, D = m->depth, nl = m->nl;
  const double *idh0 = m->idh0, *idh1 = m->idh1;
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      if (nl > 1) {
        int l = 0;
        FL(sl, l, D)[c] = add * FL(sl, l, D)[c] +
                          fac * FL(&m->strl, l, D)[c] * (FL(pl, l + 1, D)[c] - FL(pl, l, D)[c]) * idh1[l];
        for (l = 1; l < nl - 1; l++)
          FL(sl, l, D)[c] = add * FL(sl, l, D)[c] +
                            fac * (FL(&m->strl, l - 1, D)[c] * (FL(pl, l - 1, D)[c] - FL(pl, l, D)[c]) * idh0[l] +
                                   FL(&m->strl, l, D)[c] * (FL(pl, l + 1, D)[c] - FL(pl, l, D)[c]) * idh1[l]);
        l = nl - 1;
        FL(sl, l, D)[c] = add * FL(sl, l, D)[c] +
                          fac * FL(&m->strl, l - 1, D)[c] * (FL(pl, l - 1, D)[c] - FL(pl, l, D)[c]) * idh0[l];
      } else
        FL(sl, 0, D)[c] = 0.;
    }
  boundary(sl);
}

/* jacobian macro, qg.h:252-262: returns -J(p,q) */
static inline double jacobian(const double *po, const double *qo, int n, int i, int j, double Delta) {
#define P(a, b) po[IDX(n, i + (a), j + (b))]
#define Q(a, b) qo[IDX(n, i + (a), j + (b))]
  return (((Q(1, 0) - Q(-1, 0)) * (P(0, 1) - P(0, -1))
         + (Q(0, -1) - Q(0, 1)) * (P(1, 0) - P(-1, 0))
         + Q(1, 0) * (P(1, 1) - P(1, -1))
         - Q(-1, 0) * (P(-1, 1) - P(-1, -1))
         - Q(0, 1) * (P(1, 1) - P(-1, 1))
         + Q(0, -1) * (P(1, -1) - P(-1, -1))
         + P(0, 1) * (Q(1, 1) - Q(-1, 1))
         - P(0, -1) * (Q(1, -1) - Q(-1, -1))
         - P(1, 0) * (Q(1, 1) - Q(1, -1))
         + P(-1, 0) * (Q(-1, 1) - Q(-1, -1)))
        / (12. * Delta * Delta));
#undef P
#undef Q
}
/* beta_effect macro, qg.h:269 */
#define BETA_EFFECT(po, n, i, j, beta, Delta) \
  ((beta) * (po[IDX(n, (i) - 1, j)] - po[IDX(n, (i) + 1, j)]) / (2 * (Delta)))

/* comp_vel (qg.h:275-283) fused with [BASILISK] timestep() (copy newqg/qg.h:202-219):
 * foreach_face: u.x on faces i=0..n, j=0..n-1; u.y on faces j=0..n, i=0..n-1 */
static double comp_vel_timestep(orc_model *m, const double *po, double dtmax) {
  int n = m->N;
  double Delta = m->L0 / n, CFL = m->p.CFL;
  dtmax /= CFL;
  for (int i = 0; i <= n; i++)
    for (int j = 0; j < n; j++) {
      double u = -1. * 0.25 * (po[IDX(n, i, j + 1)] - po[IDX(n, i, j - 1)] +
                               po[IDX(n, i - 1, j + 1)] - po[IDX(n, i - 1, j - 1)]) / Delta;
      if (u != 0.) { double dt = Delta / fabs(u); if (dt < dtmax) dtmax = dt; }
    }
  for (int i = 0; i < n; i++)
    for (int j = 0; j <= n; j++) {
      double u = 1. * 0.25 * (po[IDX(n, i + 1, j)] - po[IDX(n, i - 1, j)] +
                              po[IDX(n, i + 1, j - 1)] - po[IDX(n, i - 1, j - 1)]) / Delta;
      if (u != 0.) { double dt = Delta / fabs(u); if (dt < dtmax) dtmax = dt; }
    }
  dtmax *= CFL;
  if (dtmax > m->ts_previous) dtmax = (m->ts_previous + 0.1 * dtmax) / 1.1;
  m->ts_previous = dtmax;
  return dtmax;
}

/* advection_pv, qg.h:287-394 (_LS_RV=1; both branches of ENERGY_CONSERV, selected by
 * m->energy_conserv) and the stochastic replacement qg_stochastic.h:17-111 (which has no
 * ENERGY_CONSERV branch).  _LS_RV=0 is the same arithmetic as flsrv = 0 (zetapl stays 0, and
 * x + jacobian(po, 0) == x).  Arguments as called from update_qg
 * (qg.h:623): qol=zeta, qotl=q, pol=psi, dqol=updates. */
static double advection_pv(orc_model *m, flist *zl, flist *qtl, flist *pl, flist *dql, double dtmax) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n, beta = m->p.beta;
  const double *idh0 = m->idh0, *idh1 = m->idh1;
  int st = m->p.stochastic;
  int ec = m->energy_conserv && !st;
  double itr = m->p.itr_stoch;
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double ju, jd;
      size_t c = IDX(n, i, j);
      if (nl > 1) {
        int l = 0;
        const double *qo = FL(zl, l, D), *po = FL(pl, l, D), *pp = FL(&m->ppl, l, D);
        const double *qot = FL(qtl, l, D), *qp = FL(&m->zetapl, l, D);
        double *dqo = FL(dql, l, D);
        const double *po2 = FL(pl, l + 1, D), *pp2 = FL(&m->ppl, l + 1, D);
        const double *s1 = FL(&m->strl, l, D), *s0;
        if (ec) { /* qg.h:310-312 */
          jd = jacobian(pp, po2, n, i, j, Delta) + jacobian(po, pp2, n, i, j, Delta);
          dqo[c] += jacobian(po, qot, n, i, j, Delta) + jacobian(pp, qo, n, i, j, Delta) +
                    BETA_EFFECT(po, n, i, j, beta, Delta) + s1[c] * jd * idh1[l];
        } else if (!st) {
          jd = jacobian(po, po2, n, i, j, Delta) + jacobian(pp, po2, n, i, j, Delta) + jacobian(po, pp2, n, i, j, Delta);
          dqo[c] += jacobian(po, qo, n, i, j, Delta) + jacobian(pp, qo, n, i, j, Delta) +
                    BETA_EFFECT(po, n, i, j, beta, Delta) + s1[c] * jd * idh1[l];
        } else {
          jd = jacobian(pp, po2, n, i, j, Delta) + jacobian(po, pp2, n, i, j, Delta);
          dqo[c] += jacobian(pp, qo, n, i, j, Delta) + BETA_EFFECT(po, n, i, j, beta, Delta) + s1[c] * jd * idh1[l];
        }
        dqo[c] += jacobian(po, qp, n, i, j, Delta);
        if (st) dqo[c] += -qot[c] * itr;
        for (l = 1; l < nl - 1; l++) {
          qo = FL(zl, l, D); po = FL(pl, l, D); qot = FL(qtl, l, D); pp = FL(&m->ppl, l, D);
          qp = FL(&m->zetapl, l, D); dqo = FL(dql, l, D);
          po2 = FL(pl, l + 1, D); pp2 = FL(&m->ppl, l + 1, D);
          s0 = FL(&m->strl, l - 1, D); s1 = FL(&m->strl, l, D);
          ju = -jd;
          if (!st && !ec)
            jd = jacobian(po, po2, n, i, j, Delta) + jacobian(pp, po2, n, i, j, Delta) + jacobian(po, pp2, n, i, j, Delta);
          else
            jd = jacobian(pp, po2, n, i, j, Delta) + jacobian(po, pp2, n, i, j, Delta);
          dqo[c] += jacobian(po, ec ? qot : qo, n, i, j, Delta) + jacobian(pp, qo, n, i, j, Delta) +
                    BETA_EFFECT(po, n, i, j, beta, Delta) + s0[c] * ju * idh0[l] + s1[c] * jd * idh1[l];
          dqo[c] += jacobian(po, qp, n, i, j, Delta);
          if (st) dqo[c] += -qot[c] * itr;
        }
        l = nl - 1;
        qo = FL(zl, l, D); po = FL(pl, l, D); qot = FL(qtl, l, D); pp = FL(&m->ppl, l, D);
        qp = FL(&m->zetapl, l, D); dqo = FL(dql, l, D);
        s0 = FL(&m->strl, l - 1, D);
        ju = -jd;
        dqo[c] += jacobian(po, ec ? qot : qo, n, i, j, Delta) + jacobian(pp, qo, n, i, j, Delta) +
                  BETA_EFFECT(po, n, i, j, beta, Delta) + s0[c] * ju * idh0[l];
        dqo[c] += jacobian(po, qp, n, i, j, Delta);
        if (st) dqo[c] += -qot[c] * itr;
      } else
        FL(dql, 0, D)[c] = 0.;
    }
  /* qg.h:383-391 */
  for (int l = 0; l < nl; l++) {
    dtmax = comp_vel_timestep(m, FL(pl, l, D), dtmax);
    dtmax = comp_vel_timestep(m, FL(&m->ppl, l, D), dtmax);
  }
  return dtmax;
}

/* dissip, qg.h:406-422 */
static void dissip(orc_model *m, flist *zl, flist *dql) {
  int n = m->N, D = m->depth, nl = m->nl;
  comp_stretch(m, zl, dql, 1., m->iRe);
  comp_del2(m, zl, &m->tmpl, 0., 1.);
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++)
        FL(dql, l, D)[IDX(n, i, j)] += FL(&m->tmpl, l, D)[IDX(n, i, j)] * m->iRe;
  comp_stretch(m, &m->tmpl, dql, 1., m->iRe4);
  comp_del2(m, &m->tmpl, dql, 1., m->iRe4);
}

/* ekman_friction qg.h:428-440; surface_forcing :446-459; qforcing :465-474;
 * bottom_topography :480-488 */
static void ekman_friction(orc_model *m, flist *zl, flist *dql) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Rom = m->p.Rom;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      FL(dql, 0, D)[c] -= m->Eks / (Rom * 2 * m->dhf[0]) * FL(zl, 0, D)[c];
      FL(dql, nl - 1, D)[c] -= m->Ekb / (Rom * 2 * m->dhf[nl - 1]) * FL(zl, nl - 1, D)[c];
    }
}
static void surface_forcing(orc_model *m, flist *dql) {
  int n = m->N, D = m->depth;
  double Delta = m->L0 / n, L0 = m->L0, Rom = m->p.Rom, tau0 = m->p.tau0;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double y = (j + 0.5) * Delta;
      FL(dql, 0, D)[IDX(n, i, j)] -= tau0 / (Rom * m->dhf[0]) * sin(2 * pi * y / L0) * sin(pi * y / L0);
    }
}
static void qforcing(orc_model *m, flist *dql) {
  int n = m->N, D = m->depth, nl = m->nl;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++)
        FL(dql, l, D)[IDX(n, i, j)] += FL(&m->q_forcl, l, D)[IDX(n, i, j)];
}
static void bottom_topography(orc_model *m, flist *pl, flist *dql) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      FL(dql, nl - 1, D)[IDX(n, i, j)] +=
          jacobian(FL(pl, nl - 1, D), FL(&m->topo, 0, D), n, i, j, Delta) /
          (FL(&m->Ro, 0, D)[IDX(n, i, j)] * m->dhf[nl - 1]);
}

/* ------------------------------------------------- poisson_layer (coupled) */
/* relax_layer, poisson_layer.h:48-150, on level l.  alpha = unity, so
 * alpha.x[1]*a[1] + alpha.x[]*a[-1] = 1.*a[1] + 1.*a[-1] (exact).
 * px,py > 1 emulates the MPI block decomposition: neighbours that belong to
 * another block are read from the pre-sweep copy `old` (the halo a rank holds
 * during a sweep); px=py=1 is the serial reference order. */
static void relax_layer_level(int nl, int l, double L0, const double *idh0, const double *idh1,
                              flist *al, flist *bl, flist *strl, int px, int py, flist *old, int colour) {
  int n = LN(l);
  double Delta = L0 / n;
  int bx = n / (px > 0 ? px : 1), by = n / (py > 0 ? py : 1);
  int blocks = (px > 1 || py > 1) && bx >= 1 && by >= 1 && old;
  if (bx < 1) bx = 1;
  if (by < 1) by = 1;
  if (blocks) fl_copy_level(old, al, l);
  if (nl <= 1) return; /* poisson_layer.h:80: no-op for nl == 1 */
#define NB(k, ii, jj, i0, j0)                                                               \
  ((blocks && ((ii) >= 0 && (ii) < n && (jj) >= 0 && (jj) < n) &&                           \
    (((ii) / bx != (i0) / bx) || ((jj) / by != (j0) / by)))                                 \
       ? FL(old, k, l)[IDX(n, ii, jj)]                                                      \
       : FL(al, k, l)[IDX(n, ii, jj)])
  /* ORC_OMP_RELAX mirrors the reference built with -fopenmp: foreach() is an
     omp-for over x, which makes the sweep thread-count dependent
     (poisson_layer.h:55-65).  Timing baseline only, never parity. */
#ifdef ORC_OMP_RELAX
#pragma omp parallel for schedule(static)
#endif
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double t0[ORC_MAXL], t1[ORC_MAXL], t2[ORC_MAXL], rhs[ORC_MAXL];
      size_t c = IDX(n, i, j);
      int ll = 0;
      if (colour >= 0 && ((i + j) & 1) != colour) continue; /* red-black: one colour per half-sweep */
      rhs[ll] = -sq(Delta) * FL(bl, ll, l)[c];
      t2[ll] = -sq(Delta) * FL(strl, ll, l)[c] * idh1[ll];
      t1[ll] = -t2[ll];
      rhs[ll] += 1. * NB(ll, i + 1, j, i, j) + 1. * NB(ll, i - 1, j, i, j); t1[ll] += 1. + 1.;
      rhs[ll] += 1. * NB(ll, i, j + 1, i, j) + 1. * NB(ll, i, j - 1, i, j); t1[ll] += 1. + 1.;
      for (ll = 1; ll < nl - 1; ll++) {
        rhs[ll] = -sq(Delta) * FL(bl, ll, l)[c];
        t0[ll] = -sq(Delta) * FL(strl, ll - 1, l)[c] * idh0[ll];
        t2[ll] = -sq(Delta) * FL(strl, ll, l)[c] * idh1[ll];
        t1[ll] = -t0[ll] - t2[ll];
        rhs[ll] += 1. * NB(ll, i + 1, j, i, j) + 1. * NB(ll, i - 1, j, i, j); t1[ll] += 1. + 1.;
        rhs[ll] += 1. * NB(ll, i, j + 1, i, j) + 1. * NB(ll, i, j - 1, i, j); t1[ll] += 1. + 1.;
      }
      ll = nl - 1;
      rhs[ll] = -sq(Delta) * FL(bl, ll, l)[c];
      t0[ll] = -sq(Delta) * FL(strl, ll - 1, l)[c] * idh0[ll];
      t1[ll] = -t0[ll];
      rhs[ll] += 1. * NB(ll, i + 1, j, i, j) + 1. * NB(ll, i - 1, j, i, j); t1[ll] += 1. + 1.;
      rhs[ll] += 1. * NB(ll, i, j + 1, i, j) + 1. * NB(ll, i, j - 1, i, j); t1[ll] += 1. + 1.;
      /* Thomas, poisson_layer.h:137-146 */
      for (ll = 1; ll < nl; ll++) {
        t1[ll] -= t0[ll] * t2[ll - 1] / t1[ll - 1];
        rhs[ll] -= t0[ll] * rhs[ll - 1] / t1[ll - 1];
      }
      FL(al, nl - 1, l)[c] = t0[nl - 1] = rhs[nl - 1] / t1[nl - 1];
      for (ll = nl - 2; ll >= 0; ll--)
        FL(al, ll, l)[c] = t0[ll] = (rhs[ll] - t2[ll] * t0[ll + 1]) / t1[ll];
    }
#undef NB
}

/* residual_layer, poisson_layer.h:157-258 (non-TREE branch), finest level.
 * face_gradient_x(a,i) = (a[i] - a[i-1])/Delta [BASILISK]. */
static double residual_layer_level(int nl, int l, double L0, const double *idh0, const double *idh1,
                                   flist *al, flist *bl, flist *resl, flist *strl) {
  int n = LN(l);
  double Delta = L0 / n, maxres = 0.;
#pragma omp parallel for schedule(static) reduction(max : maxres)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      for (int k = 0; k < nl; k++) {
        const double *a1 = FL(al, k, l);
        double r;
        if (k == 0)
          r = FL(bl, k, l)[c] + FL(strl, k, l)[c] * (a1[c] - FL(al, k + 1, l)[c]) * idh1[k];
        else if (k < nl - 1)
          r = FL(bl, k, l)[c] + FL(strl, k - 1, l)[c] * (a1[c] - FL(al, k - 1, l)[c]) * idh0[k] -
              FL(strl, k, l)[c] * (FL(al, k + 1, l)[c] - a1[c]) * idh1[k];
        else
          r = FL(bl, k, l)[c] + FL(strl, k - 1, l)[c] * (a1[c] - FL(al, k - 1, l)[c]) * idh0[k];
        r += (1. * ((a1[c] - a1[IDX(n, i - 1, j)]) / Delta) - 1. * ((a1[IDX(n, i + 1, j)] - a1[c]) / Delta)) / Delta;
        r += (1. * ((a1[c] - a1[IDX(n, i, j - 1)]) / Delta) - 1. * ((a1[IDX(n, i, j + 1)] - a1[c]) / Delta)) / Delta;
        FL(resl, k, l)[c] = r;
        if (fabs(r) > maxres) maxres = fabs(r);
      }
    }
  boundary_level(resl, l);
  return maxres;
}

/* [BASILISK] poisson.h relax()/residual() for a scalar Helmholtz problem
 * (lambda field, alpha = unity); older in-tree copy mspg/elliptic.h:265-359.
 * residual uses the face-gradient form of current Basilisk, the form
 * residual_layer was derived from. */
static void relax_scalar_level(int l, double L0, double *a, const double *b, const double *lam, int colour) {
  int n = LN(l);
  double Delta = L0 / n;
#ifdef ORC_OMP_RELAX
#pragma omp parallel for schedule(static)
#endif
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      if (colour >= 0 && ((i + j) & 1) != colour) continue;
      double nn = -sq(Delta) * b[c], d = -lam[c] * sq(Delta);
      nn += 1. * a[IDX(n, i + 1, j)] + 1. * a[IDX(n, i - 1, j)]; d += 1. + 1.;
      nn += 1. * a[IDX(n, i, j + 1)] + 1. * a[IDX(n, i, j - 1)]; d += 1. + 1.;
      a[c] = nn / d;
    }
}
static double residual_scalar_level(int l, double L0, const double *a, const double *b, double *res, const double *lam) {
  int n = LN(l);
  double Delta = L0 / n, maxres = 0.;
#pragma omp parallel for schedule(static) reduction(max : maxres)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      double r = b[c] - lam[c] * a[c];
      r += (1. * ((a[c] - a[IDX(n, i - 1, j)]) / Delta) - 1. * ((a[IDX(n, i + 1, j)] - a[c]) / Delta)) / Delta;
      r += (1. * ((a[c] - a[IDX(n, i, j - 1)]) / Delta) - 1. * ((a[IDX(n, i, j + 1)] - a[c]) / Delta)) / Delta;
      res[c] = r;
      if (fabs(r) > maxres) maxres = fabs(r);
    }
  return maxres;
}

/* [BASILISK] mg_cycle + mg_solve (poisson.h); in-tree copy
 * mspg/elliptic.h:43-99,145-229.  minlevel = 1 (poisson_layer.h:297 and
 * poisson(): max(1, p.minlevel)), NITERMAX=100, NITERMIN=1, nrelax starts 4. */
typedef struct {
  orc_model *m;
  int scalar_mode; /* 0: layer-coupled; 1: scalar helmholtz for mode `mode` */
  int mode;
} mgctx;

/* One relaxation sweep.  smoother == 0: the reference's lexicographic in-place sweep.  smoother == 1 ("rb"): the SAME
 * cell update (poisson_layer.h:80-146 / [BASILISK] relax()) applied to the cells with (i + j) even, then boundary_level,
 * then to the cells with (i + j) odd.  Cells of one colour only read cells of the other colour, so a half-sweep does
 * not depend on the traversal order, the thread count or a domain decomposition -- the dependence the reference
 * documents for its own sweep at poisson_layer.h:55-65 is removed; the iterate differs from the lexicographic one at
 * the level of the solver tolerance. */
static void mg_relax(mgctx *c, flist *da, flist *res, int l, flist *old) {
  orc_model *m = c->m;
  if (m->smoother == 1) {
    for (int colour = 0; colour < 2; colour++) {
      if (!c->scalar_mode)
        relax_layer_level(m->nl, l, m->L0, m->idh0, m->idh1, da, res, &m->strl, 1, 1, NULL, colour);
      else
        relax_scalar_level(l, m->L0, FL(da, 0, l), FL(res, 0, l), FL(&m->iBul, c->mode, l), colour);
      if (colour == 0) boundary_level(da, l);
    }
    return;
  }
  if (!c->scalar_mode) {
    int px = m->p.px, py = m->p.py;
    if (LN(l) < m->agg_n) px = py = 1;
    relax_layer_level(m->nl, l, m->L0, m->idh0, m->idh1, da, res, &m->strl, px, py, old, -1);
  } else
    relax_scalar_level(l, m->L0, FL(da, 0, l), FL(res, 0, l), FL(&m->iBul, c->mode, l), -1);
}
static double mg_residual(mgctx *c, flist *a, flist *b, flist *res) {
  orc_model *m = c->m;
  if (!c->scalar_mode)
    return residual_layer_level(m->nl, m->depth, m->L0, m->idh0, m->idh1, a, b, res, &m->strl);
  double r = residual_scalar_level(m->depth, m->L0, FL(a, 0, m->depth), FL(b, 0, m->depth),
                                   FL(res, 0, m->depth), FL(&m->iBul, c->mode, m->depth));
  boundary(res);
  return r;
}

static void mg_cycle(mgctx *c, flist *a, flist *res, flist *da, flist *old, int nrelax, int minlevel, int maxlevel) {
  restriction(res);
  if (minlevel > maxlevel) minlevel = maxlevel;
  for (int l = minlevel; l <= maxlevel; l++) {
    int n = LN(l);
    if (l == minlevel) {
      for (int k = 0; k < da->nf; k++)
        for (int i = 0; i < n; i++)
          for (int j = 0; j < n; j++) FL(da, k, l)[IDX(n, i, j)] = 0.;
    } else
      prolong_level(da, l);
    boundary_level(da, l);
    for (int i = 0; i < nrelax; i++) {
      mg_relax(c, da, res, l, old);
      boundary_level(da, l);
    }
  }
  int n = LN(maxlevel);
  for (int k = 0; k < a->nf; k++) {
    double *s = FL(a, k, maxlevel);
    const double *ds = FL(da, k, maxlevel);
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) s[IDX(n, i, j)] += ds[IDX(n, i, j)];
  }
  boundary(a);
}

/* sched != NULL: exactly ncycles cycles, cycle k with sched[k] sweeps per level, no tolerance stop and no adaptation;
 * resa_out[k] is the residual after cycle k */
static orc_mgstats mg_solve(mgctx *c, flist *a, flist *b, double tolerance, const int *sched, int ncycles, double *resa_out) {
  orc_model *m = c->m;
  int D = m->depth, n = m->N;
  flist da = fl_new(a->nf, a->bc, D);   /* homogeneous version of a's BC: same */
  flist res = fl_new(b->nf, b->bc, D);
  flist old = fl_new(a->nf, a->bc, D);
  orc_mgstats s;
  memset(&s, 0, sizeof(s));
  double sum = 0.;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int k = 0; k < b->nf; k++) sum += FL(b, k, D)[IDX(n, i, j)];
  s.sum = sum;
  s.nrelax = 4;
  double resb;
  resb = s.resb = s.resa = mg_residual(c, a, b, &res);
  for (s.i = 0; sched ? s.i < ncycles : s.i < 100 && (s.i < 1 || s.resa > tolerance); s.i++) {
    if (sched) s.nrelax = sched[s.i];
    mg_cycle(c, a, &res, &da, &old, s.nrelax, 1, D);
    s.resa = mg_residual(c, a, b, &res);
    if (sched) resa_out[s.i] = s.resa;
    else if (s.resa > tolerance) {
      if (resb / s.resa < 1.2 && s.nrelax < 100) s.nrelax++;
      else if (resb / s.resa > 10 && s.nrelax > 2) s.nrelax--;
    }
    resb = s.resa;
  }
  m->total_cycles += s.i;
  fl_free(&da); fl_free(&res); fl_free(&old);
  return s;
}

/* invertq, qg.h:113-163 */
static void invertq(orc_model *m, flist *pl, flist *ql) {
  int n = m->N, D = m->depth, nl = m->nl;
  mgctx c; c.m = m; c.scalar_mode = 0; c.mode = 0;
  if (m->p.mode_pv_invert) {
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        size_t cc = IDX(n, i, j);
        for (int mm = 0; mm < nl; mm++) {
          double *qm = FL(&m->qom, mm, D);
          qm[cc] = 0.;
          for (int l = 0; l < nl; l++) qm[cc] += FL(&m->cl2m, mm * nl + l, D)[cc] * FL(ql, l, D)[cc];
        }
      }
    boundary(&m->qom);
    for (int l = 0; l < nl; l++) {
      flist pm = m->pom, qm = m->qom; /* views on one scalar */
      pm.nf = 1; pm.d = m->pom.d + l * (D + 1);
      qm.nf = 1; qm.d = m->qom.d + l * (D + 1);
      /* poisson(): restriction({alpha,lambda}) [BASILISK] */
      flist lam = m->iBul; lam.nf = 1; lam.d = m->iBul.d + l * (D + 1);
      restriction(&lam);
      c.scalar_mode = 1; c.mode = l;
      m->mgmode[l] = m->mgpsi = mg_solve(&c, &pm, &qm, 1e-3, NULL, 0, NULL);
    }
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        size_t cc = IDX(n, i, j);
        for (int l = 0; l < nl; l++) {
          double *po = FL(pl, l, D);
          po[cc] = 0.;
          for (int mm = 0; mm < nl; mm++) po[cc] += FL(&m->cm2l, l * nl + mm, D)[cc] * FL(&m->pom, mm, D)[cc];
        }
      }
  } else {
    /* poisson_layer, poisson_layer.h:263-306: restriction(strl) every call */
    restriction(&m->strl);
    m->mgpsi = mg_solve(&c, pl, ql, 1e-3, NULL, 0, NULL);
  }
  boundary(pl);
}
void orc_invertq(orc_model *m) { invertq(m, &m->pol, &m->qol); }
int orc_test_cycles(orc_model *m, int mode, const int *nrelax, int ncycles, double *resa) {
  if (mode < -1 || mode >= m->nl || (mode >= 0 && !m->p.mode_pv_invert) || ncycles < 1 || !nrelax || !resa) return -1;
  for (int k = 0; k < ncycles; k++)
    if (nrelax[k] < 2 || nrelax[k] > 100) return -1;
  mgctx c; c.m = m; c.scalar_mode = 0; c.mode = 0;
  if (mode < 0) {
    restriction(&m->strl); /* as invertq */
    mg_solve(&c, &m->pol, &m->qol, 1e-3, nrelax, ncycles, resa);
    boundary(&m->pol);
    return 0;
  }
  const int D = m->depth;
  flist pm = m->pom, qm = m->qom, lam = m->iBul; /* views on plane `mode` */
  pm.nf = qm.nf = lam.nf = 1;
  pm.d = m->pom.d + mode * (D + 1); qm.d = m->qom.d + mode * (D + 1); lam.d = m->iBul.d + mode * (D + 1);
  restriction(&lam);
  c.scalar_mode = 1; c.mode = mode;
  mg_solve(&c, &pm, &qm, 1e-3, nrelax, ncycles, resa);
  return 0;
}
orc_mgstats orc_last_mgstats(orc_model *m, int mode) { return mode < 0 ? m->mgpsi : m->mgmode[mode]; }
int orc_total_cycles(orc_model *m) { return m->total_cycles; }

/* comp_q, qg.h:396-403 */
static void comp_q(orc_model *m, flist *pl, flist *ql) {
  comp_del2(m, pl, ql, 0., 1.);
  comp_stretch(m, pl, ql, 1., 1.);
  boundary(ql);
}
void orc_comp_q(orc_model *m) { comp_q(m, &m->pol, &m->qol); }

/* ----------------------------------------------------------- eigmod */
typedef void (*dgeev_fn)(const char *, const char *, const int *, double *, const int *, double *,
                         double *, double *, const int *, double *, const int *, double *,
                         const int *, int *, size_t, size_t);
static dgeev_fn load_dgeev(void) {
  static dgeev_fn fn = NULL;
  static int tried = 0;
  if (tried) return fn;
  tried = 1;
  const char *lib = getenv("MSQG_ORACLE_LAPACK");
  void *h = lib ? dlopen(lib, RTLD_NOW | RTLD_GLOBAL) : NULL;
  if (!h) h = dlopen("liblapack.so.3", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return NULL;
  fn = (dgeev_fn)dlsym(h, "scipy_dgeev_");
  if (!fn) fn = (dgeev_fn)dlsym(h, "dgeev_");
  return fn;
}
struct array_i { double data; int index; };
static int compare_i(const void *a, const void *b) {
  double x = ((const struct array_i *)a)->data, y = ((const struct array_i *)b)->data;
  return (x > y) - (x < y);
}
/* eigmod body for one column, eigmode.h:74-266.  LAPACKE_dgeev(ROW_MAJOR) is
 * dgeev on the transposed copy with vl/vr transposed back. */
int orc_eigmod_column(int nl, const double *dhf, const double *Fr, double Ro,
                      double *cl2m, double *cm2l, double *iBu) {
  dgeev_fn dgeev = load_dgeev();
  if (!dgeev) return -2;
  double dhc[ORC_MAXL];
  for (int l = 0; l < nl - 1; l++) dhc[l] = 0.5 * (dhf[l] + dhf[l + 1]);
  double *amat = (double *)calloc((size_t)nl * nl, sizeof(double));
  double *acm = (double *)calloc((size_t)nl * nl, sizeof(double));
  double *vl = (double *)calloc((size_t)nl * nl, sizeof(double));
  double *vr = (double *)calloc((size_t)nl * nl, sizeof(double));
  double *vlc = (double *)calloc((size_t)nl * nl, sizeof(double));
  double *vrc = (double *)calloc((size_t)nl * nl, sizeof(double));
  double *tmp = (double *)calloc((size_t)nl * nl, sizeof(double));
  double wr[ORC_MAXL], wi[ORC_MAXL];
  struct array_i wr2[ORC_MAXL];
  if (nl > 1) {
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
  double *work = (double *)calloc((size_t)lwork, sizeof(double));
  dgeev("V", "V", &nl, acm, &nl, wr, wi, vlc, &nl, vrc, &nl, work, &lwork, &info, 1, 1);
  free(work);
  for (int r = 0; r < nl; r++)
    for (int c = 0; c < nl; c++) { vl[r * nl + c] = vlc[r + nl * c]; vr[r * nl + c] = vrc[r + nl * c]; }
  if (info < 0) return -1;
  for (int l = 0; l < nl; l++) { wr2[l].data = wr[l]; wr2[l].index = l; }
  qsort(wr2, nl, sizeof(struct array_i), compare_i);
  for (int l = 0; l < nl; l++) wr[l] = wr2[l].data;
  memcpy(tmp, vr, sizeof(double) * nl * nl);
  for (int mm = 0; mm < nl; mm++)
    for (int k = 0; k < nl; k++) vr[k * nl + mm] = tmp[k * nl + wr2[mm].index];
  memcpy(tmp, vl, sizeof(double) * nl * nl);
  for (int mm = 0; mm < nl; mm++)
    for (int k = 0; k < nl; k++) vl[k * nl + mm] = tmp[k * nl + wr2[mm].index];
  double htotal = 1.;
  for (int mm = 0; mm < nl; mm++) {
    double dotp = 0.;
    for (int k = 0; k < nl; k++) dotp += dhf[k] * vr[k * nl + mm] * vr[k * nl + mm];
    double flfac = (vr[mm] > 0 ? 1 : -1) * sqrt(htotal / dotp);
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
  free(amat); free(acm); free(vl); free(vr); free(vlc); free(vrc); free(tmp);
  return 0;
}

/* eigmod, eigmode.h:65-308: per column */
static int eigmod(orc_model *m) {
  int n = m->N, D = m->depth, nl = m->nl;
  double cl[ORC_MAXL * ORC_MAXL], cm[ORC_MAXL * ORC_MAXL], ib[ORC_MAXL], fr[ORC_MAXL];
  double last_ro = 0., last_fr[ORC_MAXL];
  int have = 0;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      double ro = FL(&m->Ro, 0, D)[c];
      for (int l = 0; l < nl - 1; l++) fr[l] = FL(&m->Frl, l, D)[c];
      /* identical inputs give identical LAPACK outputs: reuse */
      int same = have && ro == last_ro;
      for (int l = 0; same && l < nl - 1; l++) same = fr[l] == last_fr[l];
      if (!same) {
        int rc = orc_eigmod_column(nl, m->dhf, fr, ro, cl, cm, ib);
        if (rc) return rc;
        have = 1; last_ro = ro; memcpy(last_fr, fr, sizeof(fr));
      }
      for (int k = 0; k < nl * nl; k++) {
        FL(&m->cl2m, k, D)[c] = cl[k];
        FL(&m->cm2l, k, D)[c] = cm[k];
      }
      for (int l = 0; l < nl; l++) FL(&m->iBul, l, D)[c] = ib[l];
    }
  boundary(&m->iBul); boundary(&m->cl2m); boundary(&m->cm2l);
  return 0;
}

/* set_const, qg.h:931-1116 (file inputs are injected through orc_set_field
 * before this call; sbc == 0 only) */
int orc_set_const(orc_model *m) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n;
  for (int l = 0; l < nl; l++) if (m->dhf[l] == 0) return -1;
  if (m->p.Rom <= 0) return -1;
  for (int l = 0; l < nl - 1; l++) m->dhc[l] = 0.5 * (m->dhf[l] + m->dhf[l + 1]);
  m->idh0[0] = 0.;
  m->idh1[0] = 1. / (m->dhc[0] * m->dhf[0]);
  for (int l = 1; l < nl - 1; l++) {
    m->idh0[l] = 1. / (m->dhc[l - 1] * m->dhf[l]);
    m->idh1[l] = 1. / (m->dhc[l] * m->dhf[l]);
  }
  m->idh0[nl - 1] = 1. / (m->dhc[nl - 2] * m->dhf[nl - 1]);
  m->idh1[nl - 1] = 0.;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double y = (j + 0.5) * Delta;
      size_t c = IDX(n, i, j);
      if (m->p.varRo > 0)
        FL(&m->Ro, 0, D)[c] = m->p.Rom / (1 + m->p.Rom * m->p.beta * (y - 0.5 * m->L0));
      else
        FL(&m->Ro, 0, D)[c] = m->p.Rom;
    }
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      for (int l = 0; l < nl - 1; l++)
        FL(&m->strl, l, D)[c] = sq(FL(&m->Frl, l, D)[c] / FL(&m->Ro, 0, D)[c]);
    }
  if (m->p.mode_pv_invert) {
    int rc = eigmod(m);
    if (rc) return rc;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        size_t c = IDX(n, i, j);
        FL(&m->sig_filt, 0, D)[c] = fmin(m->p.afilt * sqrt(-1 / FL(&m->iBul, 1, D)[c]), m->p.Lfmax);
      }
  } else
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        size_t c = IDX(n, i, j);
        FL(&m->sig_filt, 0, D)[c] = fmin(m->p.afilt * FL(&m->Rd, 0, D)[c], m->p.Lfmax);
      }
  /* filter length scale and wavelet coefficients, qg.h:1063-1090 */
  restriction(&m->sig_filt);
  for (int l = D; l >= 0; l--) { /* low pass filter */
    int nn = LN(l);
    double Dl = m->L0 / nn;
    double *sl = FL(&m->sig_lev, 0, l);
    const double *sf = FL(&m->sig_filt, 0, l);
    for (int i = 0; i < nn; i++)
      for (int j = 0; j < nn; j++) {
        double ref_flag = 0;
        if (l < D) {
          const double *ch = FL(&m->sig_lev, 0, l + 1);
          for (int a = 0; a < 2; a++)
            for (int b = 0; b < 2; b++) ref_flag += ch[IDX(2 * nn, 2 * i + a, 2 * j + b)];
        }
        size_t c = IDX(nn, i, j);
        if (ref_flag > 0) sl[c] = 1;
        else if (sf[c] > 2 * Dl) sl[c] = 0;
        else if (sf[c] <= 2 * Dl && sf[c] > Dl) sl[c] = 1 - (sf[c] - Dl) / Dl;
        else sl[c] = 1;
      }
    boundary_level(&m->sig_lev, l);
  }
  for (int l = D; l >= 0; l--) { /* high pass filter */
    int nn = LN(l);
    double *sl = FL(&m->sig_lev, 0, l);
    for (int i = 0; i < nn; i++)
      for (int j = 0; j < nn; j++) sl[IDX(nn, i, j)] = 1 - sl[IDX(nn, i, j)];
    boundary_level(&m->sig_lev, l);
  }
  comp_q(m, &m->pol, &m->qol);
  if (m->p.flsrv == 1) comp_del2(m, &m->ppl, &m->zetapl, 0., 1.0);
  /* boundary(all), qg.h:1103 */
  boundary(&m->pol); boundary(&m->qol); boundary(&m->ppl); boundary(&m->zetal);
  boundary(&m->zetapl); boundary(&m->q_forcl); boundary(&m->tmpl); boundary(&m->Frl);
  boundary(&m->strl); boundary(&m->Ro); boundary(&m->Rd); boundary(&m->topo);
  if (m->p.mode_pv_invert) { boundary(&m->pom); boundary(&m->qom); }
  if (m->p.stochastic) { boundary(&m->s_stochl); boundary(&m->n_stochl); }
  return 0;
}

/* init event, qg.c:53-70: noise() = 1 - 2*rand()/RAND_MAX [BASILISK] */
void orc_init_noise(orc_model *m, unsigned seed) {
  int n = m->N, D = m->depth, nl = m->nl;
  srand(seed);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++)
        FL(&m->pol, l, D)[IDX(n, i, j)] = 1e-3 * (1. - 2. * rand() / (double)RAND_MAX);
  orc_remove_mean_psi(m);
  if (m->p.nptr > 0) { /* qg.c:75-84 (no ptr0.bas): the same rand() stream continues */
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++)
        for (int k = 0; k < m->ptracersl.nf; k++)
          FL(&m->ptracersl, k, D)[IDX(n, i, j)] = 1e-3 * (1. - 2. * rand() / (double)RAND_MAX);
    boundary(&m->ptracersl);
  }
}
/* qg.c:66-72 with [BASILISK] statsf: sum += dv()*f, volume += dv() */
void orc_remove_mean_psi(orc_model *m) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n;
  for (int l = 0; l < nl; l++) {
    double *po = FL(&m->pol, l, D);
    double sum = 0., volume = 0.;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) { volume += sq(Delta); sum += sq(Delta) * po[IDX(n, i, j)]; }
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) po[IDX(n, i, j)] -= sum / volume;
  }
  boundary(&m->pol);
}

/* ptr_rhs, qg.h:573-588: advection + diffusion + relaxation of the passive tracers */
static void ptr_rhs(orc_model *m, flist *ptl, flist *pl, flist *dpl) {
  int n = m->N, D = m->depth, nl = m->nl, nptr = m->p.nptr;
  double Delta = m->L0 / n;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        const double *po = FL(pl, l, D);
        for (int nt = 0; nt < nptr; nt++) {
          const double *ptracers = FL(ptl, l * nptr + nt, D), *ptr_relax = FL(&m->ptr_relaxl, l * nptr + nt, D);
          double *dpdt = FL(dpl, l * nptr + nt, D);
          size_t c = IDX(n, i, j);
          dpdt[c] += jacobian(po, ptracers, n, i, j, Delta) + m->p.iPe[nt] * LAP(ptracers, n, i, j, Delta)
                     + m->p.ptr_ir[nt] * (ptr_relax[c] - ptracers[c]);
        }
      }
}

/* ------------------------------------------------------- time stepping */
/* update_qg, qg.h:609-650 */
static double update_qg(orc_model *m, flist *evolving, flist *updates, double dtmax) {
  int n = m->N, D = m->depth, nl = m->nl;
  for (int k = 0; k < nl; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) FL(updates, k, D)[IDX(n, i, j)] = 0.;
  invertq(m, &m->pol, evolving);
  comp_del2(m, &m->pol, &m->zetal, 0., 1.0);
  dtmax = advection_pv(m, &m->zetal, evolving, &m->pol, updates, dtmax);
  dissip(m, &m->zetal, updates);
  ekman_friction(m, &m->zetal, updates);
  surface_forcing(m, updates);
  qforcing(m, updates);
  if (m->flag_topo) bottom_topography(m, &m->pol, updates);
  if (m->p.nptr > 0) { /* qg.h:634-647: the tracers are the tail of `evolving`, their tendencies the tail of `updates` */
    flist *ptr = (evolving == &m->qpred) ? &m->ptr_pred : &m->ptracersl;
    for (int k = 0; k < m->dptrl.nf; k++) /* updates were zeroed at :611-613 */
      for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) FL(&m->dptrl, k, D)[IDX(n, i, j)] = 0.;
    ptr_rhs(m, ptr, &m->pol, &m->dptrl);
  }
  return dtmax;
}
double orc_update(orc_model *m, double dtmax) { return update_qg(m, &m->qol, &m->dql, dtmax); }

/* normal_noise, qg_stochastic.h:9 ; generate_noise :117-126 */
/* counter-based generator of the production noise mode (not in the reference, which draws libc rand() sequentially):
 * Philox4x32-10 (Salmon et al. 2011), counter = (cell-layer index, draw number), key = (seed, tag); the same Box-Muller
 * transform as normal_noise (qg_stochastic.h:9) on two 64-bit uniforms.  Mirrors k_noise_philox of the CUDA library. */
static void philox4x32_10(unsigned int c[4], unsigned int k0, unsigned int k1) {
  for (int r = 0; r < 10; r++) {
    unsigned long long p0 = 0xD2511F53ull * c[0], p1 = 0xCD9E8D57ull * c[2];
    unsigned int hi0 = (unsigned int)(p0 >> 32), lo0 = (unsigned int)p0, hi1 = (unsigned int)(p1 >> 32), lo1 = (unsigned int)p1;
    unsigned int n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
void orc_test_philox(unsigned int *c4, unsigned int k0, unsigned int k1) { philox4x32_10(c4, k0, k1); }
static void generate_noise(orc_model *m) {
  int n = m->N, D = m->depth, nl = m->nl;
  if (m->noise_mode == 1) {
    for (int l = 0; l < nl; l++)
      for (int j = 0; j < n; j++)
        for (int i = 0; i < n; i++) {
          unsigned long long idx = ((unsigned long long)l * n + j) * n + i;
          unsigned int c[4] = {(unsigned int)idx, (unsigned int)(idx >> 32), (unsigned int)m->noise_draw, (unsigned int)(m->noise_draw >> 32)};
          philox4x32_10(c, m->noise_seed, 0x6d737167u);
          double u1 = (((double)c[0]) * 4294967296. + (double)c[1] + 0.5) * (1. / 18446744073709551616.);
          double u2 = (((double)c[2]) * 4294967296. + (double)c[3] + 0.5) * (1. / 18446744073709551616.);
          double g = sqrt(-2. * log(u1)) * cos(2 * pi * u2);
          FL(&m->n_stochl, l, D)[IDX(n, i, j)] = m->p.amp_stoch * FL(&m->s_stochl, l, D)[IDX(n, i, j)] * g;
        }
    m->noise_draw++;
    return;
  }
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        double g = sqrt(-2. * log(((double)(rand()) + 1.) / ((double)(RAND_MAX) + 2.))) *
                   cos(2 * pi * rand() / (double)RAND_MAX);
        FL(&m->n_stochl, l, D)[IDX(n, i, j)] = m->p.amp_stoch * FL(&m->s_stochl, l, D)[IDX(n, i, j)] * g;
      }
}

/* advance_qg, qg.h:594-606 ; stochastic variant qg_stochastic.h:128-149 */
static void advance_qg(orc_model *m, flist *out, flist *in, flist *upd, double dt) {
  int n = m->N, D = m->depth, nl = m->nl;
  if (!m->p.stochastic) {
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++)
        for (int l = 0; l < nl; l++)
          FL(out, l, D)[IDX(n, i, j)] = FL(in, l, D)[IDX(n, i, j)] + FL(upd, l, D)[IDX(n, i, j)] * dt;
  } else {
    m->corrector_step = (m->corrector_step + 1) % 2;
    float dts = sqrt(dt);
    if (m->corrector_step) {
      generate_noise(m);
      dts = dts / sqrt(2);
    }
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++)
        for (int l = 0; l < nl; l++)
          FL(out, l, D)[IDX(n, i, j)] = FL(in, l, D)[IDX(n, i, j)] + FL(upd, l, D)[IDX(n, i, j)] * dt +
                                        FL(&m->n_stochl, l, D)[IDX(n, i, j)] * dts;
  }
  boundary(out);
  if (m->p.nptr > 0) { /* qg.h:597-603 runs over (nptr+1)*nl scalars (the stochastic variant, qg_stochastic.h:139-147,
                          only over nl: tracers are not supported together with -D_STOCHASTIC there either) */
    flist *pto = (out == &m->qpred) ? &m->ptr_pred : &m->ptracersl;
    flist *pti = (in == &m->qpred) ? &m->ptr_pred : &m->ptracersl;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++)
        for (int k = 0; k < pto->nf; k++)
          FL(pto, k, D)[IDX(n, i, j)] = FL(pti, k, D)[IDX(n, i, j)] + FL(&m->dptrl, k, D)[IDX(n, i, j)] * dt;
    boundary(pto);
  }
}

/* one iteration of [BASILISK] predictor-corrector.h run() given dt */
static void rk2_rest(orc_model *m, double dt) {
  advance_qg(m, &m->qpred, &m->qol, &m->dql, dt / 2.);
  update_qg(m, &m->qpred, &m->dql, dt);
  advance_qg(m, &m->qol, &m->qol, &m->dql, dt);
}
double orc_step(orc_model *m) {
  double dt = update_qg(m, &m->qol, &m->dql, m->p.DT);
  rk2_rest(m, dt);
  m->t += dt; m->iter++; m->dt = dt;
  return dt;
}
double orc_time(orc_model *m) { return m->t; }

/* writestdout, qg.c:101-109 */
double orc_ke1(orc_model *m) {
  int n = m->N, D = m->depth;
  double Delta = m->L0 / n, ke = 0;
  const double *po = FL(&m->pol, 0, D);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) ke -= 0.5 * po[IDX(n, i, j)] * LAP(po, n, i, j, Delta) * sq(Delta);
  return ke;
}

/* .bas files, auxiliar_input.h:101-149 (output_matrixl), :24-59 (input_matrixl) */
int orc_write_bas(const char *name, int nf, int N, double L0, const double *v) {
  FILE *fp = fopen(name, "w");
  if (!fp) return -1;
  float fn = N, Delta = L0 / fn;
  for (int k = 0; k < nf; k++) {
    fwrite(&fn, sizeof(float), 1, fp);
    for (int j = 0; j < N; j++) { float yp = Delta * j + 0. + Delta / 2.; fwrite(&yp, sizeof(float), 1, fp); }
    for (int i = 0; i < N; i++) {
      float xp = Delta * i + 0. + Delta / 2.;
      fwrite(&xp, sizeof(float), 1, fp);
      for (int j = 0; j < N; j++) {
        float f = v[(size_t)N * N * k + (size_t)N * j + i];
        fwrite(&f, sizeof(float), 1, fp);
      }
    }
  }
  fclose(fp);
  return 0;
}
int orc_read_bas(const char *name, int nf, int N, double L0, double *v) {
  FILE *fp = fopen(name, "r");
  if (!fp) return -1;
  double Delta = L0 / N;
  for (int k = 0; k < nf; k++) {
    float width = 0;
    if (fread(&width, sizeof(float), 1, fp) != 1) { fclose(fp); return -2; }
    int pn = (int)width;
    float *buf = (float *)malloc(sizeof(float) * (size_t)pn * pn);
    float *skip = (float *)malloc(sizeof(float) * (size_t)pn);
    if (fread(skip, sizeof(float), pn, fp) != (size_t)pn) { fclose(fp); return -2; }
    for (int i = 0; i < pn; i++) {
      float xp;
      if (fread(&xp, sizeof(float), 1, fp) != 1) { fclose(fp); return -2; }
      if (fread(buf + (size_t)i * pn, sizeof(float), pn, fp) != (size_t)pn) { fclose(fp); return -2; }
    }
    for (int i = 0; i < N; i++)
      for (int j = 0; j < N; j++) {
        double x = (i + 0.5) * Delta, y = (j + 0.5) * Delta;
        int ii = (x - 0.) * width / L0, jj = (y - 0.) * width / L0;
        v[(size_t)N * N * k + (size_t)N * j + i] =
            (ii >= 0 && ii < width && jj >= 0 && jj < width) ? buf[(size_t)ii * pn + jj] : 0.;
      }
    free(buf); free(skip);
  }
  fclose(fp);
  return 0;
}

/* [BASILISK] run() of predictor-corrector.h with the events of qg.c:
 * writestdout (i++), output (t=0; t<=tend+1e-10; t+=dtout), and dtnext(). */
static void energy_tend(orc_model *m, flist *pl, double dt, double ediag);
static void reset_layer_var(orc_model *m, flist *f);
static void filter_de(orc_model *m, flist *pml, double dtflt, double ediag);
static void wavelet_filter(orc_model *m, flist *ql, flist *pl, flist *qofl, double dtflt, int nbar);
int orc_run(orc_model *m, int max_steps, int write_files, const char *outdir, int verbose) {
  double ev_t = 0.;
  int ev_alive = 1, steps = 0;
  /* filter (t = dtflt; t <= tend+1e-10; t += dtflt), qg.h:655-658 and qg_energy.h:270-273 */
  double ev_f = m->p.dtflt;
  int evf_alive = (m->p.dtflt > 0) && (ev_f <= m->p.tend + 1e-10);
  size_t sz = (size_t)m->nl * m->N * m->N;
  double *buf = write_files ? (double *)malloc(sizeof(double) * sz) : NULL;
  char name[512];
  while (1) {
    if (evf_alive && fabs(m->t - ev_f) <= TEPS * m->t) {
      if (verbose) fprintf(stdout, "Filter solution\n");
      wavelet_filter(m, &m->qol, &m->pol, &m->qofl, m->p.dtflt, m->nbar);
      if (m->p.ediag > -1) filter_de(m, &m->po_mft, m->p.dtflt, (double)m->p.ediag);
      ev_f += m->p.dtflt;
      if (!(ev_f <= m->p.tend + 1e-10)) evf_alive = 0;
    }
    /* comp_diag (i++), qg_energy.h:289-291: defined before qg.c's events, so it runs first; `dt` is [BASILISK]'s
       global, 1. before the first step (common.h) */
    if (m->p.ediag > -1) energy_tend(m, &m->pol, m->iter == 0 ? 1. : m->dt, (double)m->p.ediag);
    if (verbose) {
      double ke = orc_ke1(m);
      fprintf(stdout, "i = %i, dt = %g, t = %g, ke_1 = %g\n", m->iter, m->dt, m->t, ke);
    }
    double tnext = HUGEV;
    if (ev_alive && fabs(m->t - ev_t) <= TEPS * m->t) {
      if (verbose) fprintf(stdout, "write file\n");
      invertq(m, &m->pol, &m->qol); /* qg.c:115 */
      if (write_files) {
        get_list(&m->pol, m->N, buf);
        snprintf(name, sizeof(name), "%s/po%09d.bas", outdir, m->iter);
        orc_write_bas(name, m->nl, m->N, m->L0, buf);
        get_list(&m->qol, m->N, buf);
        snprintf(name, sizeof(name), "%s/qo%09d.bas", outdir, m->iter);
        orc_write_bas(name, m->nl, m->N, m->L0, buf);
      }
      if (m->p.ediag > -1) { /* qg.c:139-166: write_field(de_*, name, 1/dtout) then reset */
        static const char *nm[6] = {"de_bf", "de_vd", "de_j1", "de_j2", "de_j3", "de_ft"};
        flist *L[6] = {&m->de_bfl, &m->de_vdl, &m->de_j1l, &m->de_j2l, &m->de_j3l, &m->de_ftl};
        double idtout = 1 / m->p.dtout;
        for (int k = 0; k < 6; k++) {
          if (write_files) {
            get_list(L[k], m->N, buf);
            for (size_t c = 0; c < sz; c++) buf[c] *= idtout;
            snprintf(name, sizeof(name), "%s/%s%09d.bas", outdir, nm[k], m->iter);
            orc_write_bas(name, m->nl, m->N, m->L0, buf);
          }
          reset_layer_var(m, L[k]);
        }
      }
      if (m->p.dtflt > 0) { /* qg.c:124-129: filtered stream function from the filter mean, then nbar = 0 */
        invertq(m, &m->tmpl, &m->qofl);
        if (write_files) {
          get_list(&m->tmpl, m->N, buf);
          snprintf(name, sizeof(name), "%s/pf%09d.bas", outdir, m->iter);
          orc_write_bas(name, m->nl, m->N, m->L0, buf);
        }
        m->nbar = 0;
      }
      if (m->p.nptr > 0 && write_files) { /* qg.c:168-171 */
        size_t szp = (size_t)m->ptracersl.nf * m->N * m->N;
        double *bp = (double *)malloc(sizeof(double) * szp);
        get_list(&m->ptracersl, m->N, bp);
        snprintf(name, sizeof(name), "%s/ptr%09d.bas", outdir, m->iter);
        orc_write_bas(name, m->ptracersl.nf, m->N, m->L0, bp);
        free(bp);
      }
      ev_t += m->p.dtout;
      if (!(ev_t <= m->p.tend + 1e-10)) ev_alive = 0;
    }
    if (!ev_alive) break;
    if (ev_t > m->t) tnext = ev_t;
    if (evf_alive && ev_f > m->t && ev_f < tnext) tnext = ev_f;
    if (max_steps >= 0 && steps >= max_steps) break;
    /* dt = dtnext(update(evolving, updates, DT)) */
    double dt = update_qg(m, &m->qol, &m->dql, m->p.DT);
    if (tnext != HUGEV && tnext > m->t) {
      unsigned int nn = (tnext - m->t) / dt;
      if (nn == 0) dt = tnext - m->t;
      else {
        double dt1 = (tnext - m->t) / nn;
        if (dt1 > dt * (1. + TEPS)) dt = (tnext - m->t) / (nn + 1);
        else if (dt1 < dt) dt = dt1;
        tnext = m->t + dt;
      }
    } else
      tnext = m->t + dt;
    rk2_rest(m, dt);
    m->dt = dt; m->t = tnext; m->iter++;
    steps++;
  }
  free(buf);
  return steps;
}

/* ----------------------------------------------------------- multi-scale wavelet filter, qg.h:509-560
 * [BASILISK] wavelet() / inverse_wavelet() (grid/multigrid-common.h), restated: the coefficient of a fine cell is
 * its value minus the bilinear prolongation of the restricted field; the root keeps the value itself. */
static inline double bilinear_at(const double *c, int nc, int i, int j) { /* fine cell (i,j), coarse array c */
  int ic = i >> 1, jc = j >> 1;
  int cx = (i & 1) ? 1 : -1, cy = (j & 1) ? 1 : -1;
  return (9. * c[IDX(nc, ic, jc)] + 3. * (c[IDX(nc, ic + cx, jc)] + c[IDX(nc, ic, jc + cy)]) + c[IDX(nc, ic + cx, jc + cy)]) / 16.;
}
static void wavelet(orc_model *m, flist *sl, int k, flist *w) {
  int D = m->depth;
  /* restriction({s}) was done for the whole list by the caller */
  for (int l = D - 1; l >= 0; l--) {
    int nf = LN(l + 1), nc = LN(l);
    const double *s = FL(sl, k, l + 1), *c = FL(sl, k, l);
    double *wf = FL(w, 0, l + 1);
    for (int i = 0; i < nf; i++)
      for (int j = 0; j < nf; j++) {
        double wv = s[IDX(nf, i, j)];
        double sp = bilinear_at(c, nc, i, j);
        wv -= sp; /* difference between fine value and its prolongation */
        wf[IDX(nf, i, j)] = wv;
      }
    boundary_level(w, l + 1);
  }
  FL(w, 0, 0)[IDX(1, 0, 0)] = FL(sl, k, 0)[IDX(1, 0, 0)]; /* root cell */
  boundary_level(w, 0);
}
static void inverse_wavelet(orc_model *m, flist *sl, int k, flist *w) {
  int D = m->depth;
  FL(sl, k, 0)[IDX(1, 0, 0)] = FL(w, 0, 0)[IDX(1, 0, 0)];
  boundary_level(sl, 0);
  for (int l = 0; l <= D - 1; l++) {
    int nf = LN(l + 1), nc = LN(l);
    double *s = FL(sl, k, l + 1);
    const double *c = FL(sl, k, l), *wf = FL(w, 0, l + 1);
    for (int i = 0; i < nf; i++)
      for (int j = 0; j < nf; j++) {
        double v = bilinear_at(c, nc, i, j);
        v += wf[IDX(nf, i, j)];
        s[IDX(nf, i, j)] = v;
      }
    boundary_level(sl, l + 1);
  }
}
/* wavelet_filter, qg.h:509-560.  nbar is passed BY VALUE in the reference (the nbar++ at :558 is lost). */
static void wavelet_filter(orc_model *m, flist *ql, flist *pl, flist *qofl, double dtflt, int nbar) {
  int n = m->N, D = m->depth, nl = m->nl;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) FL(&m->tmpl, l, D)[IDX(n, i, j)] = FL(ql, l, D)[IDX(n, i, j)];
  invertq(m, pl, ql);
  restriction(pl);
  for (int k = 0; k < nl; k++) {
    wavelet(m, pl, k, &m->wvl);
    for (int l = 0; l <= D; l++) {
      int nn = LN(l);
      double *w = FL(&m->wvl, 0, l);
      const double *sg = FL(&m->sig_lev, 0, l);
      for (int i = 0; i < nn; i++)
        for (int j = 0; j < nn; j++) w[IDX(nn, i, j)] *= sg[IDX(nn, i, j)];
      boundary_level(&m->wvl, l);
    }
    inverse_wavelet(m, pl, k, &m->wvl);
  }
  comp_q(m, pl, ql);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        size_t c = IDX(n, i, j);
        double *qof = FL(qofl, l, D);
        qof[c] = (qof[c] * nbar + (FL(&m->tmpl, l, D)[c] - FL(ql, l, D)[c]) / dtflt) / (nbar + 1);
      }
  if (dtflt < 0.0) /* for energy diag: restore qo to prefiltered value */
    fl_copy_level(ql, &m->tmpl, D); /* list_copy_deep(tmpl, qol, nl) */
  boundary(qofl);
}
void orc_get_siglev(orc_model *m, int level, double *v) {
  int nn = LN(level);
  for (int i = 0; i < nn; i++)
    for (int j = 0; j < nn; j++) v[(size_t)nn * j + i] = FL(&m->sig_lev, 0, level)[IDX(nn, i, j)];
}
void orc_wavelet_filter(orc_model *m, double dtflt) { wavelet_filter(m, &m->qol, &m->pol, &m->qofl, dtflt, m->nbar); }

/* ----------------------------------------------------------- energy diagnostics, msqg/qg_energy.h
 * "We multiply all terms of the PV equation by -po*dt" (:1-5).  _LS_RV = 1; the ENERGY_CONSERV branch of
 * advection_de (:33-35, :64-66, :100-102, :132-134) is selected by m->energy_conserv. */
static void set_vars_energy(orc_model *m) { /* qg_energy.h:244-253 */
  if (m->energy_vars) return;
  flist *L[8] = {&m->de_bfl, &m->de_vdl, &m->de_j1l, &m->de_j2l, &m->de_j3l, &m->de_ftl, &m->tmp2l, &m->po_mft};
  for (int k = 0; k < 8; k++) *L[k] = create_layer_var(m->nl, 0, m->depth);
  m->nme_ft = 0;
  m->energy_vars = 1;
}
static void reset_layer_var(orc_model *m, flist *f) { /* layer.h:37-41 */
  int n = m->N, D = m->depth;
  for (int l = 0; l < f->nf; l++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) FL(f, l, D)[IDX(n, i, j)] = 0.;
}
void orc_reset_energy(orc_model *m) {
  set_vars_energy(m);
  flist *L[6] = {&m->de_bfl, &m->de_vdl, &m->de_j1l, &m->de_j2l, &m->de_j3l, &m->de_ftl};
  for (int k = 0; k < 6; k++) reset_layer_var(m, L[k]);
}
/* advection_de, qg_energy.h:28-154; called with qol = zetal (:231) */
static void advection_de(orc_model *m, flist *ql, flist *pl, double dt, double ediag) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n, beta = m->p.beta;
  const double *idh0 = m->idh0, *idh1 = m->idh1;
  const int ec = m->energy_conserv;
  if (ec) comp_q(m, pl, &m->tmp2l); /* qg_energy.h:33-35 */
#define JC(a, b) jacobian(a, b, n, i, j, Delta)
#define QT(l) FL(&m->tmp2l, l, D)
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      double ju_1, jd_1, ju_2, jd_2, ju_3, jd_3, jc;
      if (nl > 1) {
        int l = 0;
        const double *qo = FL(ql, l, D), *po = FL(pl, l, D), *pp = FL(&m->ppl, l, D), *qp = FL(&m->zetapl, l, D);
        const double *po2 = FL(pl, l + 1, D), *pp2 = FL(&m->ppl, l + 1, D);
        const double *s1 = FL(&m->strl, l, D), *s0;
        double *de_j1 = FL(&m->de_j1l, l, D), *de_j2 = FL(&m->de_j2l, l, D), *de_j3 = FL(&m->de_j3l, l, D);
        jd_1 = JC(po, po2);
        jd_2 = JC(pp, po2);
        jd_3 = JC(po, pp2);
        jc = JC(po, pp);
        if (ec) de_j1[c] += (JC(po, QT(l))) * dt * (-po[c] * (1 - ediag) + ediag);
        else de_j1[c] += (JC(po, qo) + s1[c] * jd_1 * idh1[l]) * dt * (-po[c] * (1 - ediag) + ediag);
        de_j2[c] += (JC(pp, qo) + s1[c] * (jd_2 + jc) * idh1[l]) * dt * (-po[c] * (1 - ediag) + ediag);
        de_j3[c] += (BETA_EFFECT(po, n, i, j, beta, Delta) + s1[c] * (jd_3 - jc) * idh1[l]) * dt * (-po[c] * (1 - ediag) + ediag);
        de_j3[c] += JC(po, qp) * dt * (-po[c] * (1 - ediag) + ediag);
        for (l = 1; l < nl - 1; l++) {
          qo = FL(ql, l, D); po = FL(pl, l, D); pp = FL(&m->ppl, l, D); qp = FL(&m->zetapl, l, D);
          po2 = FL(pl, l + 1, D); pp2 = FL(&m->ppl, l + 1, D);
          de_j1 = FL(&m->de_j1l, l, D); de_j2 = FL(&m->de_j2l, l, D); de_j3 = FL(&m->de_j3l, l, D);
          s0 = FL(&m->strl, l - 1, D); s1 = FL(&m->strl, l, D);
          ju_1 = -jd_1;
          ju_2 = -jd_3; /* swap */
          ju_3 = -jd_2; /* swap */
          jd_1 = JC(po, po2);
          jd_2 = JC(pp, po2);
          jd_3 = JC(po, pp2);
          jc = JC(po, pp);
          if (ec) de_j1[c] += (JC(po, QT(l))) * dt * (-po[c] * (1 - ediag) + ediag);
          else de_j1[c] += (JC(po, qo) + s0[c] * ju_1 * idh0[l] + s1[c] * jd_1 * idh1[l]) * dt * (-po[c] * (1 - ediag) + ediag);
          de_j2[c] += (JC(pp, qo) + s0[c] * (ju_2 + jc) * idh0[l] + s1[c] * (jd_2 + jc) * idh1[l]) * dt * (-po[c] * (1 - ediag) + ediag);
          de_j3[c] += (BETA_EFFECT(po, n, i, j, beta, Delta) + s0[c] * (ju_3 - jc) * idh0[l] + s1[c] * (jd_3 - jc) * idh1[l]) * dt * (-po[c] * (1 - ediag) + ediag);
          de_j3[c] += JC(po, qp) * dt * (-po[c] * (1 - ediag) + ediag);
        }
        l = nl - 1;
        qo = FL(ql, l, D); po = FL(pl, l, D); pp = FL(&m->ppl, l, D); qp = FL(&m->zetapl, l, D);
        de_j1 = FL(&m->de_j1l, l, D); de_j2 = FL(&m->de_j2l, l, D); de_j3 = FL(&m->de_j3l, l, D);
        s0 = FL(&m->strl, l - 1, D);
        ju_1 = -jd_1;
        ju_2 = -jd_3; /* swap */
        ju_3 = -jd_2; /* swap */
        jc = JC(po, pp);
        if (ec) de_j1[c] += (JC(po, QT(l))) * dt * (-po[c] * (1 - ediag) + ediag);
        else de_j1[c] += (JC(po, qo) + s0[c] * ju_1 * idh0[l]) * dt * (-po[c] * (1 - ediag) + ediag);
        de_j2[c] += (JC(pp, qo) + s0[c] * (ju_2 + jc) * idh0[l]) * dt * (-po[c] * (1 - ediag) + ediag);
        de_j3[c] += (BETA_EFFECT(po, n, i, j, beta, Delta) + s0[c] * (ju_3 - jc) * idh0[l]) * dt * (-po[c] * (1 - ediag) + ediag);
        de_j3[c] += JC(po, qp) * dt * (-po[c] * (1 - ediag) + ediag);
      } else {
        FL(&m->de_j1l, 0, D)[c] = 0; FL(&m->de_j2l, 0, D)[c] = 0; FL(&m->de_j3l, 0, D)[c] = 0;
      }
    }
#undef JC
#undef QT
}
/* dissip_de, qg_energy.h:157-187 */
static void dissip_de(orc_model *m, flist *zl, flist *dql, flist *pl, double dt, double ediag) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Delta = m->L0 / n;
  comp_del2(m, zl, &m->tmpl, 0., 1.);
  comp_stretch(m, zl, &m->tmp2l, 0., 1.);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        size_t c = IDX(n, i, j);
        double *dqo = FL(dql, l, D);
        const double *p4 = FL(&m->tmpl, l, D), *str = FL(&m->tmp2l, l, D), *po = FL(pl, l, D);
        dqo[c] += (p4[c] + str[c]) * m->iRe * dt * (-po[c] * (1 - ediag) + ediag);
        dqo[c] += m->iRe4 * LAP(p4, n, i, j, Delta) * dt * (-po[c] * (1 - ediag) + ediag);
      }
  comp_stretch(m, &m->tmpl, &m->tmp2l, 0., 1.);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        size_t c = IDX(n, i, j);
        double *dqo = FL(dql, l, D);
        const double *str = FL(&m->tmp2l, l, D), *po = FL(pl, l, D);
        dqo[c] += m->iRe4 * (str[c]) * dt * (-po[c] * (1 - ediag) + ediag);
      }
}
/* ekman_friction_de, qg_energy.h:189-204 */
static void ekman_friction_de(orc_model *m, flist *zl, flist *dql, flist *pl, double dt, double ediag) {
  int n = m->N, D = m->depth, nl = m->nl;
  double Rom = m->p.Rom;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      size_t c = IDX(n, i, j);
      FL(dql, 0, D)[c] -= m->Eks / (Rom * 2 * m->dhf[0]) * FL(zl, 0, D)[c] * dt * (-FL(pl, 0, D)[c] * (1 - ediag) + ediag);
      FL(dql, nl - 1, D)[c] -= m->Ekb / (Rom * 2 * m->dhf[nl - 1]) * FL(zl, nl - 1, D)[c] * dt * (-FL(pl, nl - 1, D)[c] * (1 - ediag) + ediag);
    }
}
/* filter_de, qg_energy.h:207-226 */
static void filter_de(orc_model *m, flist *pml, double dtflt, double ediag) {
  int n = m->N, D = m->depth, nl = m->nl;
  set_vars_energy(m);
  wavelet_filter(m, &m->qol, &m->pol, &m->tmp2l, -dtflt, 0);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        size_t c = IDX(n, i, j);
        double *pm = FL(pml, l, D);
        FL(&m->de_ftl, l, D)[c] += FL(&m->tmp2l, l, D)[c] * dtflt * (-pm[c] * (1 - ediag) + ediag);
        pm[c] = 0;
      }
  m->nme_ft = 0;
}
/* energy_tend, qg_energy.h:228-242 */
static void energy_tend(orc_model *m, flist *pl, double dt, double ediag) {
  int n = m->N, D = m->depth, nl = m->nl;
  set_vars_energy(m);
  comp_del2(m, pl, &m->zetal, 0., 1.0);
  advection_de(m, &m->zetal, pl, dt, ediag);
  dissip_de(m, &m->zetal, &m->de_vdl, pl, dt, ediag);
  ekman_friction_de(m, &m->zetal, &m->de_bfl, pl, dt, ediag);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++)
      for (int l = 0; l < nl; l++) {
        size_t c = IDX(n, i, j);
        double *pm = FL(&m->po_mft, l, D);
        pm[c] = (pm[c] * m->nme_ft + FL(pl, l, D)[c]) / (m->nme_ft + 1);
      }
  m->nme_ft += 1;
}
void orc_filter_de(orc_model *m, double dtflt) { filter_de(m, &m->po_mft, dtflt, (double)m->p.ediag); }
void orc_energy_tend(orc_model *m, double dt) { energy_tend(m, &m->pol, dt, (double)m->p.ediag); }
/* pystep_de, qg_energy.h:294-340: ediag = 1, dt = 1 (locals shadow the globals).  filter_de is called with pol in
 * the po_mft slot (:330), so psi is zeroed on the way out; with the default dtflt = -1 the inner wavelet_filter sees
 * +1 and leaves q filtered. */
void orc_pystep_de(orc_model *m, const double *po_py, double *de_bf, double *de_vd, double *de_j1, double *de_j2,
                   double *de_j3, double *de_ft, int onlyKE) {
  int n = m->N, D = m->depth, nl = m->nl;
  double ediag = 1., dt = 1.;
  set_list(&m->pol, n, po_py);
  orc_reset_energy(m);
  comp_del2(m, &m->pol, &m->zetal, 0., 1.0);
  comp_q(m, &m->pol, &m->qol);
  if (onlyKE == 1)
    for (int l = 0; l < nl - 1; l++)
      for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) FL(&m->strl, l, D)[IDX(n, i, j)] = 0.;
  advection_de(m, &m->zetal, &m->pol, dt, ediag);
  dissip_de(m, &m->zetal, &m->de_vdl, &m->pol, dt, ediag);
  ekman_friction_de(m, &m->zetal, &m->de_bfl, &m->pol, dt, ediag);
  filter_de(m, &m->pol, m->p.dtflt, ediag);
  get_list(&m->de_bfl, n, de_bf); get_list(&m->de_vdl, n, de_vd);
  get_list(&m->de_j1l, n, de_j1); get_list(&m->de_j2l, n, de_j2);
  get_list(&m->de_j3l, n, de_j3); get_list(&m->de_ftl, n, de_ft);
}

/* python entry points, qg_bfn.h:21-103 */
void orc_pystep_bfn(orc_model *m, const double *q_in, double *tend, double direction, int vartype) {
  double dtmax = m->p.DT;
  double Re = m->p.Re, Re4 = m->p.Re4;
  if (direction > 0) {
    m->iRe = (Re == 0) ? 0. : 1 / Re;
    m->iRe4 = (Re4 == 0) ? 0. : -1 / Re4;
    m->Eks = fabs(m->Eks); m->Ekb = fabs(m->Ekb);
  } else {
    m->iRe = (Re == 0) ? 0. : -1 / Re;
    m->iRe4 = (Re4 == 0) ? 0. : 1 / Re4;
    m->Eks = -fabs(m->Eks); m->Ekb = -fabs(m->Ekb);
  }
  int n = m->N, D = m->depth;
  for (int k = 0; k < m->nl; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) FL(&m->dql, k, D)[IDX(n, i, j)] = 0.;
  if (vartype == 1) {
    set_list(&m->qol, n, q_in);
    invertq(m, &m->pol, &m->qol);
    comp_del2(m, &m->pol, &m->zetal, 0., 1.0);
    dtmax = advection_pv(m, &m->zetal, &m->qol, &m->pol, &m->dql, dtmax);
    dissip(m, &m->zetal, &m->dql);
    ekman_friction(m, &m->zetal, &m->dql);
    surface_forcing(m, &m->dql);
    if (m->flag_topo) bottom_topography(m, &m->pol, &m->dql);
    get_list(&m->dql, n, tend);
  }
  (void)dtmax;
}
void orc_pyq2p(orc_model *m, double *po, const double *qo) {
  int n = m->N, D = m->depth;
  for (int k = 0; k < m->nl; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) FL(&m->pol, k, D)[IDX(n, i, j)] = 0.;
  set_list(&m->qol, n, qo);
  invertq(m, &m->pol, &m->qol);
  get_list(&m->pol, n, po);
}
void orc_pyp2q(orc_model *m, const double *po, double *qo) {
  int n = m->N, D = m->depth;
  for (int k = 0; k < m->nl; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) FL(&m->qol, k, D)[IDX(n, i, j)] = 0.;
  set_list(&m->pol, n, po);
  comp_q(m, &m->pol, &m->qol);
  get_list(&m->qol, n, qo);
}

/* --------------------------------------------------- unit-level hooks */
static void metrics(int nl, const double *dh, double *idh0, double *idh1) {
  double dhc[ORC_MAXL];
  for (int l = 0; l < nl - 1; l++) dhc[l] = 0.5 * (dh[l] + dh[l + 1]);
  idh0[0] = 0.; idh1[0] = 1. / (dhc[0] * dh[0]);
  for (int l = 1; l < nl - 1; l++) { idh0[l] = 1. / (dhc[l - 1] * dh[l]); idh1[l] = 1. / (dhc[l] * dh[l]); }
  idh0[nl - 1] = 1. / (dhc[nl - 2] * dh[nl - 1]); idh1[nl - 1] = 0.;
}
static void load_level(flist *f, int l, const double *v) {
  int n = LN(l);
  for (int k = 0; k < f->nf; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) FL(f, k, l)[IDX(n, i, j)] = v[(size_t)n * n * k + (size_t)n * j + i];
  boundary_level(f, l);
}
static void store_level(const flist *f, int l, double *v) {
  int n = LN(l);
  for (int k = 0; k < f->nf; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) v[(size_t)n * n * k + (size_t)n * j + i] = FL(f, k, l)[IDX(n, i, j)];
}
void orc_test_relax(int nl, int level, double L0, const double *dh, const double *s,
                    double *a, const double *b, int nsweeps, int px, int py) {
  double idh0[ORC_MAXL], idh1[ORC_MAXL];
  metrics(nl, dh, idh0, idh1);
  flist A = fl_new(nl, BC_DIRICHLET0, level), B = fl_new(nl, BC_DIRICHLET0, level);
  flist S = fl_new(nl, BC_NEUMANN, level), O = fl_new(nl, BC_DIRICHLET0, level);
  load_level(&A, level, a); load_level(&B, level, b);
  S.nf = nl - 1; load_level(&S, level, s); S.nf = nl;
  for (int k = 0; k < nsweeps; k++) {
    if (px < 0) { /* red-black ordering (orc_test_relax_rb) */
      relax_layer_level(nl, level, L0, idh0, idh1, &A, &B, &S, 1, 1, NULL, 0);
      boundary_level(&A, level);
      relax_layer_level(nl, level, L0, idh0, idh1, &A, &B, &S, 1, 1, NULL, 1);
    } else
      relax_layer_level(nl, level, L0, idh0, idh1, &A, &B, &S, px, py, &O, -1);
    boundary_level(&A, level);
  }
  store_level(&A, level, a);
  fl_free(&A); fl_free(&B); fl_free(&S); fl_free(&O);
}
void orc_test_relax_rb(int nl, int level, double L0, const double *dh, const double *s,
                       double *a, const double *b, int nsweeps) {
  orc_test_relax(nl, level, L0, dh, s, a, b, nsweeps, -1, -1);
}
double orc_test_residual(int nl, int level, double L0, const double *dh, const double *s,
                         const double *a, const double *b, double *res) {
  double idh0[ORC_MAXL], idh1[ORC_MAXL];
  metrics(nl, dh, idh0, idh1);
  flist A = fl_new(nl, BC_DIRICHLET0, level), B = fl_new(nl, BC_DIRICHLET0, level);
  flist S = fl_new(nl, BC_NEUMANN, level), R = fl_new(nl, BC_DIRICHLET0, level);
  load_level(&A, level, a); load_level(&B, level, b);
  S.nf = nl - 1; load_level(&S, level, s); S.nf = nl;
  double r = residual_layer_level(nl, level, L0, idh0, idh1, &A, &B, &R, &S);
  store_level(&R, level, res);
  fl_free(&A); fl_free(&B); fl_free(&S); fl_free(&R);
  return r;
}
void orc_test_restrict(int nf, int level, const double *fine, double *coarse) {
  flist F = fl_new(nf, BC_DIRICHLET0, level);
  load_level(&F, level, fine);
  int n = LN(level - 1), nf2 = 2 * n;
  for (int k = 0; k < nf; k++)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        const double *a = FL(&F, k, level);
        double sum = 0.;
        sum += a[IDX(nf2, 2 * i, 2 * j)]; sum += a[IDX(nf2, 2 * i, 2 * j + 1)];
        sum += a[IDX(nf2, 2 * i + 1, 2 * j)]; sum += a[IDX(nf2, 2 * i + 1, 2 * j + 1)];
        FL(&F, k, level - 1)[IDX(n, i, j)] = sum / 4;
      }
  store_level(&F, level - 1, coarse);
  fl_free(&F);
}
void orc_test_prolong(int nf, int level, const double *coarse, double *fine) {
  flist F = fl_new(nf, BC_DIRICHLET0, level);
  load_level(&F, level - 1, coarse);
  prolong_level(&F, level);
  store_level(&F, level, fine);
  fl_free(&F);
}
static void test_relax_scalar(int level, double L0, const double *lam, double *a, const double *b, int nsweeps, int rb);
void orc_test_relax_scalar(int level, double L0, const double *lam, double *a, const double *b, int nsweeps) {
  test_relax_scalar(level, L0, lam, a, b, nsweeps, 0);
}
void orc_test_relax_scalar_rb(int level, double L0, const double *lam, double *a, const double *b, int nsweeps) {
  test_relax_scalar(level, L0, lam, a, b, nsweeps, 1);
}
static void test_relax_scalar(int level, double L0, const double *lam, double *a, const double *b, int nsweeps, int rb) {
  flist A = fl_new(1, BC_DIRICHLET0, level), B = fl_new(1, BC_DIRICHLET0, level), Lm = fl_new(1, BC_NEUMANN, level);
  load_level(&A, level, a); load_level(&B, level, b); load_level(&Lm, level, lam);
  for (int k = 0; k < nsweeps; k++) {
    if (rb) {
      relax_scalar_level(level, L0, FL(&A, 0, level), FL(&B, 0, level), FL(&Lm, 0, level), 0);
      boundary_level(&A, level);
      relax_scalar_level(level, L0, FL(&A, 0, level), FL(&B, 0, level), FL(&Lm, 0, level), 1);
    } else
      relax_scalar_level(level, L0, FL(&A, 0, level), FL(&B, 0, level), FL(&Lm, 0, level), -1);
    boundary_level(&A, level);
  }
  store_level(&A, level, a);
  fl_free(&A); fl_free(&B); fl_free(&Lm);
}
double orc_test_residual_scalar(int level, double L0, const double *lam, const double *a, const double *b, double *res) {
  flist A = fl_new(1, BC_DIRICHLET0, level), B = fl_new(1, BC_DIRICHLET0, level), Lm = fl_new(1, BC_NEUMANN, level);
  flist R = fl_new(1, BC_DIRICHLET0, level);
  load_level(&A, level, a); load_level(&B, level, b); load_level(&Lm, level, lam);
  double r = residual_scalar_level(level, L0, FL(&A, 0, level), FL(&B, 0, level), FL(&R, 0, level), FL(&Lm, 0, level));
  store_level(&R, level, res);
  fl_free(&A); fl_free(&B); fl_free(&Lm); fl_free(&R);
  return r;
}
