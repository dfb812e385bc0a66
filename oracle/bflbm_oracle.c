/* TEST INFRASTRUCTURE ONLY -- the checker, never the product.
 *
 * Plain-C restatement of the reference's fluctuating binary D3Q19 step
 * (LBM_d3q19.H / LBM_binary.H of MDProject/Binary-Fluctuating-Lattice-Boltzmann).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference leg may load it.  It exists because /root/reference (and
 * therefore a rebuild of oracle/_ref) is not available on the GPU box.
 *
 * It is written independently of the reference's data structures (no ghost
 * cells, periodic index wrap, no FillBoundary) but keeps the reference's
 * floating-point operation ORDER expression by expression, so that -- compiled
 * with -ffp-contract=off like oracle/_ref -- it reproduces the reference
 * bit for bit.  tests/test_oracle.py pins it against oracle/_ref (when present)
 * and against the committed fixtures in tests/golden/ generated from oracle/_ref.
 *
 * Parity status: deterministic path (kBT = 0, or injected normals) PINNED by
 * those fixtures.  The reference's Gaussian stream (amrex::RandomNormal) is
 * third-party and unpinned (SURVEY.md 8(c)); normals are therefore an INPUT
 * here (33 per cell in the reference's draw order, LBM_binary.H:115-127).
 */
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define NVEL 19

/* LBM_d3q19.H:12-32 */
static const int C[NVEL][3] = {
    {0, 0, 0},  {1, 0, 0},  {-1, 0, 0}, {0, 1, 0},  {0, -1, 0}, {0, 0, 1},  {0, 0, -1},
    {1, 1, 0},  {-1, -1, 0}, {1, -1, 0}, {-1, 1, 0}, {0, 1, 1},  {0, -1, -1}, {0, 1, -1},
    {0, -1, 1}, {1, 0, 1},  {-1, 0, -1}, {1, 0, -1}, {-1, 0, 1}};
/* LBM_d3q19.H:34-54, 56-76 (filled in oracle_create so the divisions are done at run time like the reference's initialisers) */
static double W[NVEL], B[NVEL];
static double cs2, cs4; /* LBM_d3q19.H:6-7 */

typedef struct {
  double kBT, tau_f, tau_g, alpha0, alpha1, kappa, rho_lo, rho_hi;
} oracle_params;

typedef struct {
  int nx, ny, nz;
  size_t n;
  oracle_params p;
  double *f, *g, *fnew, *gnew; /* [19][n] */
  double *h;                   /* hydrovs    [22][n] */
  double *hb;                  /* hydrovsbar [9][n]  */
  double *fn, *gn;             /* noise      [19][n] */
  const double* normals;       /* injected standard normals, 33 per cell, or NULL (= 0) */
  /* USE_REF_STATE (LBM_binary.H:12, 92-107): noise amplitudes from the equilibrium profiles, shifted by the integer part of
   * (centre of mass - com_ref); NULL = the shipped build (current densities) */
  double *rho_eq, *phi_eq, *rhot_eq; /* [n] each */
  double com_ref[3];
  /* set_ref_shift: the shift the next noise generations use instead of (int)(com - com_ref), so that an oracle on a window of a
   * larger box can take that box's shift; force_shift = 0 (the default) computes it as the reference does */
  int force_shift, forced_shift[3];
} oracle_lattice;

static void init_constants(void) {
  cs2 = 1. / 3.;
  cs4 = (1. / 3.) * (1. / 3.);
  W[0] = 1. / 3.;
  for (int i = 1; i <= 6; ++i) W[i] = 1. / 18.;
  for (int i = 7; i < NVEL; ++i) W[i] = 1. / 36.;
  const double b[NVEL] = {1.0,     1. / 3., 1. / 3., 1. / 3., 2. / 3., 4. / 3., 4. / 9., 1. / 9., 1. / 9., 1. / 9.,
                          2. / 3., 2. / 3., 2. / 3., 2. / 9., 2. / 9., 2. / 9., 2.0,     4. / 3., 4. / 9.};
  memcpy(B, b, sizeof(B));
}

/* forward transform m = M f; LBM_d3q19.H:100-156 */
static void moments19(const double* fs, double* m) {
  double f, mc0, mc1, mc2, mx1, my1, mz1, mx2, my2, mz2, mx3, my3, mz3;
  double mxy, mxz, myz, mxx1, myy1, mzz1, mxx2, myy2, mzz2;
  f = fs[0]; mc0 = f;
  f = fs[1]; mx1 = f; mxx1 = f;
  f = fs[2]; mx1 -= f; mxx1 += f;
  f = fs[3]; my1 = f; myy1 = f;
  f = fs[4]; my1 -= f; myy1 += f;
  f = fs[5]; mz1 = f; mzz1 = f;
  f = fs[6]; mz1 -= f; mzz1 += f;
  f = fs[7]; mx2 = f; my3 = f; mxy = f; mxx2 = f;
  f = fs[8]; mx2 -= f; my3 -= f; mxy += f; mxx2 += f;
  f = fs[9]; mx2 += f; my3 -= f; mxy -= f; mxx2 += f;
  f = fs[10]; mx2 -= f; my3 += f; mxy -= f; mxx2 += f;
  f = fs[11]; my2 = f; mz3 = f; myz = f; myy2 = f;
  f = fs[12]; my2 -= f; mz3 -= f; myz += f; myy2 += f;
  f = fs[13]; my2 += f; mz3 -= f; myz -= f; myy2 += f;
  f = fs[14]; my2 -= f; mz3 += f; myz -= f; myy2 += f;
  f = fs[15]; mz2 = f; mx3 = f; mxz = f; mzz2 = f;
  f = fs[16]; mz2 -= f; mx3 -= f; mxz += f; mzz2 += f;
  f = fs[17]; mz2 -= f; mx3 += f; mxz -= f; mzz2 += f;
  f = fs[18]; mz2 += f; mx3 -= f; mxz -= f; mzz2 += f;
  mc1 = mxx1 + myy1 + mzz1;
  mc2 = mxx2 + myy2 + mzz2;
  m[0] = mc0 + mc1 + mc2;
  m[1] = mx1 + mx2 + mx3;
  m[2] = my1 + my2 + my3;
  m[3] = mz1 + mz2 + mz3;
  m[4] = mc2 - mc0;
  m[5] = 3. * mxx1 - mc1 + mc2 - 3. * myy2;
  m[6] = myy1 - mzz1 + mxx2 - mzz2;
  m[7] = mxy;
  m[8] = myz;
  m[9] = mxz;
  m[10] = m[1] - 3. * mx1;
  m[11] = m[2] - 3. * my1;
  m[12] = m[3] - 3. * mz1;
  m[13] = mx2 - mx3;
  m[14] = my2 - my3;
  m[15] = mz2 - mz3;
  m[16] = m[0] - 3. * mc1;
  m[17] = mc1 - 3. * mxx1 + mc2 - 3. * myy2;
  m[18] = mzz1 - myy1 + mxx2 - mzz2;
}

/* inverse transform f = M^-1 m; LBM_d3q19.H:167-247 */
static void populations19(const double* mom, double* f) {
  static const double div[NVEL] = {36., 12., 12., 12., 24., 48., 16., 4., 4., 4., 24., 24., 24., 8., 8., 8., 72., 48., 16.};
  double m[NVEL];
  for (int a = 0; a < NVEL; ++a) m[a] = mom[a] / div[a];
  const double mc0 = 12. * (m[0] - m[4] + m[16]);
  const double mc1 = 2. * (m[0] - 2. * m[16]);
  const double mc2 = m[0] + m[4] + m[16];
  const double mx1 = 2. * (m[1] - 2. * m[10]);
  const double my1 = 2. * (m[2] - 2. * m[11]);
  const double mz1 = 2. * (m[3] - 2. * m[12]);
  const double mx2 = m[1] + m[10] + m[13];
  const double my2 = m[2] + m[11] + m[14];
  const double mz2 = m[3] + m[12] + m[15];
  const double mx3 = m[1] + m[10] - m[13];
  const double my3 = m[2] + m[11] - m[14];
  const double mz3 = m[3] + m[12] - m[15];
  const double mxx1 = mc1 + 4. * (m[5] - m[17]);
  const double myy1 = mc1 - 2. * (m[5] - m[6]) + 2. * (m[17] - m[18]);
  const double mzz1 = mc1 - 2. * (m[5] + m[6]) + 2. * (m[17] + m[18]);
  const double mxy2 = mc2 + (m[5] + m[6]) + (m[17] + m[18]);
  const double mxz2 = mc2 + (m[5] - m[6]) + (m[17] - m[18]);
  const double myz2 = mc2 - 2. * (m[5] + m[17]);
  const double mxy = m[7], myz = m[8], mxz = m[9];
  f[0] = mc0;
  f[1] = mxx1 + mx1;
  f[2] = mxx1 - mx1;
  f[3] = myy1 + my1;
  f[4] = myy1 - my1;
  f[5] = mzz1 + mz1;
  f[6] = mzz1 - mz1;
  f[7] = mxy2 + mx2 + my3 + mxy;
  f[8] = mxy2 - mx2 - my3 + mxy;
  f[9] = mxy2 + mx2 - my3 - mxy;
  f[10] = mxy2 - mx2 + my3 - mxy;
  f[11] = myz2 + my2 + mz3 + myz;
  f[12] = myz2 - my2 - mz3 + myz;
  f[13] = myz2 + my2 - mz3 - myz;
  f[14] = myz2 - my2 + mz3 - myz;
  f[15] = mxz2 + mz2 + mx3 + mxz;
  f[16] = mxz2 - mz2 - mx3 + mxz;
  f[17] = mxz2 - mz2 + mx3 - mxz;
  f[18] = mxz2 + mz2 - mx3 - mxz;
}

/* LBM_binary.H:356-402 */
static void equilibrium_moments(double dens, const double* u, double* mEq) {
  const double coefA = dens, coefB = 1., coefAB = coefA * coefB, coefC = 1. / cs2;
  double AD[3][3];
  AD[0][0] = (coefA * u[0] * u[0]) / 2. / cs4;
  AD[0][1] = (coefA * u[0] * u[1]) / 2. / cs4;
  AD[0][2] = (coefA * u[0] * u[2]) / 2. / cs4;
  AD[1][0] = AD[0][1];
  AD[1][1] = (coefA * u[1] * u[1]) / 2. / cs4;
  AD[1][2] = (coefA * u[1] * u[2]) / 2. / cs4;
  AD[2][0] = AD[0][2];
  AD[2][1] = AD[1][2];
  AD[2][2] = (coefA * u[2] * u[2]) / 2. / cs4;
  const double tr = AD[0][0] + AD[1][1] + AD[2][2];
  mEq[0] = coefAB;
  mEq[1] = coefC * cs2 * (coefA * u[0]);
  mEq[2] = coefC * cs2 * (coefA * u[1]);
  mEq[3] = coefC * cs2 * (coefA * u[2]);
  mEq[4] = 2. * cs4 * tr;
  mEq[5] = 6. * cs4 * AD[0][0] - 2. * cs4 * tr;
  mEq[6] = 2. * cs4 * (AD[1][1] - AD[2][2]);
  mEq[7] = cs4 * (AD[0][1] + AD[1][0]);
  mEq[8] = cs4 * (AD[1][2] + AD[2][1]);
  mEq[9] = cs4 * (AD[0][2] + AD[2][0]);
  for (int a = 10; a < NVEL; ++a) mEq[a] = 0.;
}

/* LBM_binary.H:404-449; note tau_f for BOTH species (:424) */
static void phi_moments(const oracle_params* p, double dens, const double* u, const double* a, double* mPhi) {
  const double coefA = dens, coefB = 0., coefAB = coefA * coefB, coefC = 1. / cs2, coefAC = coefA * coefC;
  double AD[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) AD[i][j] = a[i] * (coefA * u[j]) / cs4;
  const double tr = AD[0][0] + AD[1][1] + AD[2][2];
  const double mod = 1. / (1. + 1. / (2. * p->tau_f));
  mPhi[0] = mod * coefAB;
  mPhi[1] = mod * coefAC * cs2 * a[0];
  mPhi[2] = mod * coefAC * cs2 * a[1];
  mPhi[3] = mod * coefAC * cs2 * a[2];
  mPhi[4] = mod * 2. * cs4 * tr;
  mPhi[5] = mod * (6. * cs4 * AD[0][0] - 2. * cs4 * tr);
  mPhi[6] = mod * 2. * cs4 * (AD[1][1] - AD[2][2]);
  mPhi[7] = mod * cs4 * (AD[0][1] + AD[1][0]);
  mPhi[8] = mod * cs4 * (AD[1][2] + AD[2][1]);
  mPhi[9] = mod * cs4 * (AD[0][2] + AD[2][0]);
  for (int k = 10; k < NVEL; ++k) mPhi[k] = 0.;
}

static inline size_t cell_index(const oracle_lattice* L, int x, int y, int z) {
  return (size_t)x + (size_t)L->nx * ((size_t)y + (size_t)L->ny * (size_t)z);
}
static inline int wrap(int i, int n) { return i < 0 ? i + n : (i >= n ? i - n : i); }

/* collide (LBM_binary.H:451-516) + push stream with periodic images (LBM_binary.H:518-531, 565-573) */
static void collide_stream_all(oracle_lattice* L) {
  const oracle_params* p = &L->p;
  const size_t n = L->n;
  const double tau_f_bar = p->tau_f * (1. + 0.5 / p->tau_f);
  const double tau_g_bar = p->tau_g * (1. + 0.5 / p->tau_g);
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
  for (int z = 0; z < L->nz; ++z)
    for (int y = 0; y < L->ny; ++y)
      for (int x = 0; x < L->nx; ++x) {
        const size_t c = cell_index(L, x, y, z);
        double fs[NVEL], gs[NVEL], mf[NVEL], mg[NVEL], mfEq[NVEL], mgEq[NVEL], mPf[NVEL], mPg[NVEL];
        const double rho = L->h[0 * n + c], phi = L->h[1 * n + c];
        const double uf[3] = {L->h[2 * n + c], L->h[3 * n + c], L->h[4 * n + c]};
        const double ug[3] = {L->h[6 * n + c], L->h[7 * n + c], L->h[8 * n + c]};
        const double af[3] = {L->h[9 * n + c], L->h[10 * n + c], L->h[11 * n + c]};
        const double ag[3] = {L->h[12 * n + c], L->h[13 * n + c], L->h[14 * n + c]};
        for (int i = 0; i < NVEL; ++i) { fs[i] = L->f[i * n + c]; gs[i] = L->g[i * n + c]; }
        moments19(fs, mf);
        moments19(gs, mg);
        double vb[3];
        for (int k = 0; k < 3; ++k) vb[k] = (rho * uf[k] + phi * ug[k]) / (rho + phi);
        equilibrium_moments(rho, vb, mfEq);
        equilibrium_moments(phi, vb, mgEq);
        phi_moments(p, rho, uf, af, mPf);
        phi_moments(p, phi, ug, ag, mPg);
        for (int a = 0; a < NVEL; ++a) {
          const double Raf = 1. / tau_f_bar * (mfEq[a] - mf[a]) + mPf[a] + L->fn[a * n + c];
          const double Rag = 1. / tau_g_bar * (mgEq[a] - mg[a]) + mPg[a] + L->gn[a * n + c];
          mf[a] = mf[a] + Raf;
          mg[a] = mg[a] + Rag;
        }
        populations19(mf, fs);
        populations19(mg, gs);
        for (int i = 0; i < NVEL; ++i) {
          const size_t t = cell_index(L, wrap(x + C[i][0], L->nx), wrap(y + C[i][1], L->ny), wrap(z + C[i][2], L->nz));
          L->fnew[i * n + t] = fs[i];
          L->gnew[i * n + t] = gs[i];
        }
      }
  double* t;
  t = L->f; L->f = L->fnew; L->fnew = t;
  t = L->g; L->g = L->gnew; L->gnew = t;
}

/* LBM_binary.H:315-354 */
static void hydrovars_density_all(oracle_lattice* L) {
  const size_t n = L->n;
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
  for (long c = 0; c < (long)n; ++c) {
    double fs[NVEL], gs[NVEL], mf[NVEL], mg[NVEL];
    double rho = 0., phi = 0.;
    for (int i = 0; i < NVEL; ++i) {
      fs[i] = L->f[i * n + c]; gs[i] = L->g[i * n + c];
      rho += fs[i]; phi += gs[i];
    }
    L->hb[0 * n + c] = rho;
    L->hb[1 * n + c] = phi;
    moments19(fs, mf);
    moments19(gs, mg);
    for (int k = 1; k <= 3; ++k) {
      L->hb[(k + 1) * n + c] = (fabs(mf[0]) > FLT_EPSILON) ? mf[k] / mf[0] : 0.;
      L->hb[(k + 5) * n + c] = (fabs(mg[0]) > FLT_EPSILON) ? mg[k] / mg[0] : 0.;
    }
    L->hb[5 * n + c] = mf[0] + mg[0];
  }
}

/* LBM_binary.H:73-132 (non-USE_REF_STATE branch); tau_g_bar := tau_f_bar (:80) */
/* update_com (LBM_hydrovs.H:26-60) of one [n] field: sum rho * index / sum rho, cells visited x fastest */
static void center_of_mass(const oracle_lattice* L, const double* rho, double* com) {
  double mass = 0., sx = 0., sy = 0., sz = 0.;
  for (int k = 0; k < L->nz; ++k)
    for (int j = 0; j < L->ny; ++j)
      for (int i = 0; i < L->nx; ++i) {
        const double r = rho[(size_t)i + (size_t)L->nx * ((size_t)j + (size_t)L->ny * (size_t)k)];
        mass += r; sx += r * i; sy += r * j; sz += r * k;
      }
  com[0] = sx / mass; com[1] = sy / mass; com[2] = sz / mass;
}

/* relative: the caller is LBM_init / LBM_timestep (pos_com - com_ref[0], LBM_binary.H:586-588, 651-653); the analytic inits
 * pass the absolute centre of mass (LBM_binary.H:623-625) */
static void thermal_noise_all(oracle_lattice* L, int relative) {
  const oracle_params* p = &L->p;
  const size_t n = L->n;
  const double tfb = 1. / (p->tau_f + 0.5), tgb = tfb, tfb2 = tfb * tfb, tgb2 = tgb * tgb;
  int shift[3] = {0, 0, 0};
  if (L->rho_eq) {
    double com[3];
    center_of_mass(L, L->hb, com);
    for (int d = 0; d < 3; ++d) shift[d] = (int)(relative ? com[d] - L->com_ref[d] : com[d]);
    if (L->force_shift)
      for (int d = 0; d < 3; ++d) shift[d] = L->forced_shift[d];
  }
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
  for (long c = 0; c < (long)n; ++c) {
    const double* N = L->normals ? L->normals + 33 * (size_t)c : NULL;
    int d = 0;
    double rho = L->hb[0 * n + c], phi = L->hb[1 * n + c], rhot = rho + phi;
    if (L->rho_eq) { /* LBM_binary.H:92-107 */
      int x = (int)(c % (size_t)L->nx), y = (int)((c / (size_t)L->nx) % (size_t)L->ny), z = (int)(c / ((size_t)L->nx * L->ny));
      int xs = x - shift[0], ys = y - shift[1], zs = z - shift[2];
      if (xs < 0) xs += L->nx;
      if (xs > L->nx - 1) xs -= L->nx;
      if (ys < 0) ys += L->ny;
      if (ys > L->ny - 1) ys -= L->ny;
      if (zs < 0) zs += L->nz;
      if (zs > L->nz - 1) zs -= L->nz;
      const size_t cs = cell_index(L, xs, ys, zs);
      rho = L->rho_eq[cs]; phi = L->phi_eq[cs]; rhot = L->rhot_eq[cs];
    }
    L->fn[0 * n + c] = 0.;
    L->gn[0 * n + c] = 0.;
    for (int a = 1; a <= 3; ++a) {
      const double z = N ? N[d] : 0.; ++d;
      L->fn[a * n + c] = sqrt(2. * (tfb - 0.5 * tfb2) * p->kBT * fabs(rho * phi / rhot)) * (0. + 1. * z);
      L->gn[a * n + c] = -L->fn[a * n + c];
    }
    for (int a = 4; a < NVEL; ++a) {
      const double z1 = N ? N[d] : 0.; ++d;
      const double z2 = N ? N[d] : 0.; ++d;
      L->fn[a * n + c] = sqrt(2. * (tfb - 0.5 * tfb2) * p->kBT / cs2 * B[a] * fabs(rho)) * (0. + 1. * z1);
      L->gn[a * n + c] = sqrt(2. * (tgb - 0.5 * tgb2) * p->kBT / cs2 * B[a] * fabs(phi)) * (0. + 1. * z2);
    }
  }
}

/* LBM_binary.H:134-150 */
static void gradient(const oracle_lattice* L, const double* field, int x, int y, int z, double* grad) {
  grad[0] = grad[1] = grad[2] = 0.;
  for (int i = 0; i < NVEL; ++i) {
    const size_t t = cell_index(L, wrap(x + C[i][0], L->nx), wrap(y + C[i][1], L->ny), wrap(z + C[i][2], L->nz));
    const double v = field[t];
    for (int dir = 0; dir < 3; ++dir) grad[dir] += W[i] / cs2 * v * C[i][dir];
  }
}

/* LBM_binary.H:196-313 */
static void hydrovars_all(oracle_lattice* L) {
  const oracle_params* p = &L->p;
  const size_t n = L->n;
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
  for (int z = 0; z < L->nz; ++z)
    for (int y = 0; y < L->ny; ++y)
      for (int x = 0; x < L->nx; ++x) {
        const size_t c = cell_index(L, x, y, z);
        double* h = L->h;
        const double rho = L->hb[0 * n + c], phi = L->hb[1 * n + c];
        double jf[3] = {0., 0., 0.}, jg[3] = {0., 0., 0.};
        h[0 * n + c] = rho;
        h[1 * n + c] = phi;
        for (int i = 0; i < NVEL; ++i) {
          const double fi = L->f[i * n + c], gi = L->g[i * n + c];
          jf[0] += fi * C[i][0]; jf[1] += fi * C[i][1]; jf[2] += fi * C[i][2];
          jg[0] += gi * C[i][0]; jg[1] += gi * C[i][1]; jg[2] += gi * C[i][2];
        }
        double grad_rho[3], grad_phi[3];
        gradient(L, L->hb + 0 * n, x, y, z, grad_rho);
        gradient(L, L->hb + 1 * n, x, y, z, grad_phi);
        double ufb[3], ugb[3], afb[3], agb[3], nfv[3], ngv[3];
        for (int k = 0; k < 3; ++k) {
          ufb[k] = (fabs(rho) > FLT_EPSILON) ? jf[k] / rho : 0.;
          ugb[k] = (fabs(phi) > FLT_EPSILON) ? jg[k] / phi : 0.;
          afb[k] = (fabs(rho) > FLT_EPSILON) ? -cs2 * p->alpha0 * rho * grad_phi[k] / rho : 0.;
          agb[k] = (fabs(phi) > FLT_EPSILON) ? -cs2 * p->alpha0 * phi * grad_rho[k] / phi : 0.;
          nfv[k] = (fabs(rho) > FLT_EPSILON) ? L->fn[(k + 1) * n + c] / rho : 0.;
          ngv[k] = (fabs(phi) > FLT_EPSILON) ? L->gn[(k + 1) * n + c] / phi : 0.;
        }
        for (int k = 0; k < 3; ++k) {
          h[(2 + k) * n + c] = ufb[k] + 0.5 * afb[k] - 0.5 / (p->tau_f + 0.5) * phi / (rho + phi) * (ufb[k] - ugb[k] + 0.5 * (afb[k] - agb[k])) + 0.5 * nfv[k];
          h[(6 + k) * n + c] = ugb[k] + 0.5 * agb[k] - 0.5 / (p->tau_g + 0.5) * rho / (rho + phi) * (ugb[k] - ufb[k] + 0.5 * (agb[k] - afb[k])) + 0.5 * ngv[k];
        }
        const double rho_tot = rho + phi;
        h[5 * n + c] = rho_tot;
        for (int k = 0; k < 3; ++k) {
          h[(9 + k) * n + c] = afb[k];
          h[(12 + k) * n + c] = agb[k];
          h[(15 + k) * n + c] = (rho * ufb[k] + phi * ugb[k] + 0.5 * (rho * afb[k] + phi * agb[k])) / rho_tot;
        }
        h[18 * n + c] = nfv[0];
        h[19 * n + c] = ngv[0];
        h[20 * n + c] = ufb[0];
        h[21 * n + c] = ugb[0];
      }
}

/* the tail every init and every step share: LBM_binary.H:583-592, 621-627 */
static void refresh_derived(oracle_lattice* L, int relative) {
  hydrovars_density_all(L);
  thermal_noise_all(L, relative);
  hydrovars_all(L);
}

/* ------------------------------- C ABI ----------------------------------- */
void* oracle_create(int nx, int ny, int nz) {
  init_constants();
  oracle_lattice* L = (oracle_lattice*)calloc(1, sizeof(oracle_lattice));
  L->nx = nx; L->ny = ny; L->nz = nz;
  L->n = (size_t)nx * ny * nz;
  const size_t n = L->n;
  L->f = (double*)calloc(NVEL * n, sizeof(double));
  L->g = (double*)calloc(NVEL * n, sizeof(double));
  L->fnew = (double*)calloc(NVEL * n, sizeof(double));
  L->gnew = (double*)calloc(NVEL * n, sizeof(double));
  L->h = (double*)calloc(22 * n, sizeof(double));
  L->hb = (double*)calloc(9 * n, sizeof(double));
  L->fn = (double*)calloc(NVEL * n, sizeof(double));
  L->gn = (double*)calloc(NVEL * n, sizeof(double));
  /* shipped defaults: LBM_d3q19.H:10, LBM_binary.H:18-30 */
  L->p.kBT = 0.; L->p.tau_f = 0.5; L->p.tau_g = 0.5; L->p.alpha0 = 4.; L->p.alpha1 = 0.; L->p.kappa = 4.;
  L->p.rho_lo = 0.; L->p.rho_hi = 1.;
  return L;
}
void oracle_destroy(void* h) {
  oracle_lattice* L = (oracle_lattice*)h;
  free(L->f); free(L->g); free(L->fnew); free(L->gnew); free(L->h); free(L->hb); free(L->fn); free(L->gn);
  free(L->rho_eq); free(L->phi_eq); free(L->rhot_eq);
  free(L);
}
void oracle_set_params(void* h, double kBT, double tau_f, double tau_g, double alpha0, double alpha1, double kappa,
                       double rho_lo, double rho_hi) {
  oracle_lattice* L = (oracle_lattice*)h;
  L->p.kBT = kBT; L->p.tau_f = tau_f; L->p.tau_g = tau_g; L->p.alpha0 = alpha0; L->p.alpha1 = alpha1;
  L->p.kappa = kappa; L->p.rho_lo = rho_lo; L->p.rho_hi = rho_hi;
}
/* equilibrium profiles of the fluctuating run (main_run_job.cpp:216-236: load, com_ref = their centres of mass); NULL = off */
void oracle_set_equilibrium(void* h, const double* rho_eq, const double* phi_eq, const double* rhot_eq) {
  oracle_lattice* L = (oracle_lattice*)h;
  free(L->rho_eq); free(L->phi_eq); free(L->rhot_eq);
  L->rho_eq = L->phi_eq = L->rhot_eq = NULL;
  if (!rho_eq) return;
  const size_t n = L->n;
  L->rho_eq = (double*)malloc(n * sizeof(double)); L->phi_eq = (double*)malloc(n * sizeof(double)); L->rhot_eq = (double*)malloc(n * sizeof(double));
  memcpy(L->rho_eq, rho_eq, n * sizeof(double)); memcpy(L->phi_eq, phi_eq, n * sizeof(double)); memcpy(L->rhot_eq, rhot_eq, n * sizeof(double));
  center_of_mass(L, L->rho_eq, L->com_ref);
}
/* the integer shift (x, y, z) of the reference-state noise for the next noise generations; NULL = computed from the centre of
 * mass again (test hook: a window of a larger box cannot compute that box's shift) */
void oracle_set_ref_shift(void* h, const int* shift3) {
  oracle_lattice* L = (oracle_lattice*)h;
  L->force_shift = shift3 != NULL;
  for (int d = 0; d < 3; ++d) L->forced_shift[d] = shift3 ? shift3[d] : 0;
}
/* 33 standard normals per cell (cell-major, reference draw order) used by the NEXT noise generation; NULL = zeros */
void oracle_set_normals(void* h, const double* normals) { ((oracle_lattice*)h)->normals = normals; }

static void fill_from_density(oracle_lattice* L, size_t c, double rho, double phi) {
  for (int i = 0; i < NVEL; ++i) {
    L->f[i * L->n + c] = W[i] * rho;
    L->g[i * L->n + c] = W[i] * phi;
  }
}
/* LBM_binary.H:598-629 */
void oracle_init_mixture(void* h) {
  oracle_lattice* L = (oracle_lattice*)h;
  const double C1 = 0.5, C2 = 0.5;
  for (size_t c = 0; c < L->n; ++c) fill_from_density(L, c, 2. * C1, 2. * C2);
  refresh_derived(L, 0);
}
/* LBM_binary.H:663-695 */
void oracle_init_stripe(void* h, double frac) {
  oracle_lattice* L = (oracle_lattice*)h;
  const oracle_params* p = &L->p;
  const double rho_t = p->rho_hi + p->rho_lo;
  const double pos_lo = (-0.5 * frac) * L->nz, pos_hi = (0.5 * frac) * L->nz;
  for (int z = 0; z < L->nz; ++z) {
    const double pos = z - L->nz / 2; /* integer division, :680 */
    const double rho = (p->rho_hi - p->rho_lo) * 0.5 * (tanh((pos - pos_lo) / sqrt(p->kappa)) + tanh((pos_hi - pos) / sqrt(p->kappa))) + p->rho_lo;
    for (int y = 0; y < L->ny; ++y)
      for (int x = 0; x < L->nx; ++x) fill_from_density(L, cell_index(L, x, y, z), rho, rho_t - rho);
  }
  refresh_derived(L, 0);
}
/* LBM_binary.H:698-742; rz uses box[0] and integer division (:725) */
void oracle_init_droplet(void* h, double r_frac) {
  oracle_lattice* L = (oracle_lattice*)h;
  const oracle_params* p = &L->p;
  const double R = r_frac * L->nx;
  for (int z = 0; z < L->nz; ++z)
    for (int y = 0; y < L->ny; ++y)
      for (int x = 0; x < L->nx; ++x) {
        const double rx = x - L->nx / 2.;
        const double ry = y - L->ny / 2.;
        const double rz = z - L->nx / 2;
        const double r2 = rx * rx + ry * ry + rz * rz;
        const double r = sqrt(r2);
        const double rho_tot = p->rho_hi + p->rho_lo;
        const double rho = (p->rho_hi - p->rho_lo) * (1. + tanh((R - r) / sqrt(p->kappa))) / 2. + p->rho_lo;
        fill_from_density(L, cell_index(L, x, y, z), rho, rho_tot - rho);
      }
  refresh_derived(L, 0);
}
/* restart entry, LBM_binary.H:631-661 */
void oracle_init_from_populations(void* h, const double* f0, const double* g0) {
  oracle_lattice* L = (oracle_lattice*)h;
  memcpy(L->f, f0, NVEL * L->n * sizeof(double));
  memcpy(L->g, g0, NVEL * L->n * sizeof(double));
  refresh_derived(L, 1);
}
/* LBM_timestep, LBM_binary.H:544-594 */
void oracle_step(void* h, int nsteps) {
  oracle_lattice* L = (oracle_lattice*)h;
  for (int s = 0; s < nsteps; ++s) {
    collide_stream_all(L);
    refresh_derived(L, 1);
  }
}
void oracle_get_populations(void* h, double* f, double* g) {
  oracle_lattice* L = (oracle_lattice*)h;
  memcpy(f, L->f, NVEL * L->n * sizeof(double));
  memcpy(g, L->g, NVEL * L->n * sizeof(double));
}
void oracle_get_hydrovars(void* h, double* out22) { oracle_lattice* L = (oracle_lattice*)h; memcpy(out22, L->h, 22 * L->n * sizeof(double)); }
void oracle_get_hydrovars_bar(void* h, double* out9) { oracle_lattice* L = (oracle_lattice*)h; memcpy(out9, L->hb, 9 * L->n * sizeof(double)); }
void oracle_get_noise(void* h, double* fn, double* gn) {
  oracle_lattice* L = (oracle_lattice*)h;
  memcpy(fn, L->fn, NVEL * L->n * sizeof(double));
  memcpy(gn, L->gn, NVEL * L->n * sizeof(double));
}
void oracle_moments(const double* f19, double* m19) { init_constants(); moments19(f19, m19); }
void oracle_populations(const double* m19, double* f19) { init_constants(); populations19(m19, f19); }
void oracle_constants(int* c57, double* w19, double* b19) {
  init_constants();
  for (int i = 0; i < NVEL; ++i) {
    for (int d = 0; d < 3; ++d) c57[3 * i + d] = C[i][d];
    w19[i] = W[i]; b19[i] = B[i];
  }
}
int oracle_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
void oracle_set_num_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}
