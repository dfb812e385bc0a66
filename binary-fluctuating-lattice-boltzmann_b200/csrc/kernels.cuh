// CUDA kernels of the fluctuating binary D3Q19 step (sm_100a).
//
// Data layout in HBM (one z-slab of the periodic box; the whole box is the slab with nzl = nz):
//   X  : double [2 species][19][nzl+2][ny][nx]   "pre-stream" populations: the post-stream population
//        f_i(x) of the reference's fold/gold equals X_i(x - c_i) (pull).  Plane 0 and nzl+1 are ghost
//        planes (neighbour slab or periodic image); x and y wrap by index arithmetic.
//   R  : double2 [nzl+2][ny][nx]                  (rho, phi) of the post-stream populations, with ghost planes
//   E  : double2 [brick][Lz+2][Ty+2][Tx+2]        per-brick partial sums of next-step (rho, phi) (fused algorithm)
// SoA per component = AMReX's own FAB order (x fastest ... component slowest).
#pragma once
#include "physics.cuh"

namespace bflbm {

struct Geom {
  int nx, ny, nzl;      // local slab (valid cells)
  int nz_global, z0;    // global box height and first global plane of the slab
  int zwrap;            // 1: whole box -- the thread-per-cell kernels wrap z by index arithmetic and never read a ghost plane
  long long plane;      // nx*ny
  long long comp;       // (nzl+2)*plane  : stride between components of X
};

__device__ __forceinline__ long long cell_global(const Geom& G, int x, int y, int zl) {
  return (long long)x + (long long)G.nx * ((long long)y + (long long)G.ny * (long long)(G.z0 + zl));
}

// Neighbour index tables of one cell: xs[c+1] = wrapped x + c, yrow[c+1] = (wrapped y + c)*nx,
// zpl[c+1] = (zl + 1 + c)*plane (ghost planes make z wrap-free).
struct CellIdx {
  int xs[3];
  long long yrow[3], zpl[3];
};
__device__ __forceinline__ CellIdx cell_idx(const Geom& G, int x, int y, int zl) {
  CellIdx I;
  I.xs[0] = (x == 0) ? G.nx - 1 : x - 1;
  I.xs[1] = x;
  I.xs[2] = (x == G.nx - 1) ? 0 : x + 1;
  I.yrow[0] = (long long)((y == 0) ? G.ny - 1 : y - 1) * G.nx;
  I.yrow[1] = (long long)y * G.nx;
  I.yrow[2] = (long long)((y == G.ny - 1) ? 0 : y + 1) * G.nx;
  I.zpl[0] = (long long)((G.zwrap && zl == 0) ? G.nzl : zl) * G.plane;
  I.zpl[1] = (long long)(zl + 1) * G.plane;
  I.zpl[2] = (long long)((G.zwrap && zl == G.nzl - 1) ? 1 : zl + 2) * G.plane;
  return I;
}
// index of the cell at (x,y,z) + s*c_i, s = +1 or -1
template <int S>
__device__ __forceinline__ long long nbr(const CellIdx& I, int i) {
  return I.zpl[1 + S * cz(i)] + I.yrow[1 + S * cy(i)] + I.xs[1 + S * cx(i)];
}

// USE_REF_STATE noise (LBM_binary.H:12, 92-107): eq = [rho_eq | phi_eq | rhot_eq], each nx*ny*nz_global doubles (the WHOLE box,
// also on a slab); shift = integer part of (centre of mass - com_ref), recomputed on the device after every step.
struct RefState {
  const double* eq;   // nullptr: the shipped behaviour (current densities)
  const int* shift;
};
// offset in one eq component of the cell (x, y, global plane z0 + zl) shifted by -s: a single periodic wrap per axis, like the
// reference (LBM_binary.H:97-102)
__device__ __forceinline__ long long ref_offset(const Geom& G, int sx, int sy, int sz, int x, int y, int zl) {
  int xs = x - sx, ys = y - sy, zs = G.z0 + zl - sz;
  if (xs < 0) xs += G.nx;
  if (xs > G.nx - 1) xs -= G.nx;
  if (ys < 0) ys += G.ny;
  if (ys > G.ny - 1) ys -= G.ny;
  if (zs < 0) zs += G.nz_global;
  if (zs > G.nz_global - 1) zs -= G.nz_global;
  return (long long)zs * G.plane + (long long)ys * G.nx + xs;
}
__device__ __forceinline__ bool ref_densities(const Geom& G, const RefState& RS, int x, int y, int zl, double (&d)[3]) {
  if (RS.eq == nullptr) return false;
  const long long n = G.plane * G.nz_global, c = ref_offset(G, RS.shift[0], RS.shift[1], RS.shift[2], x, y, zl);
  d[0] = RS.eq[c];
  d[1] = RS.eq[n + c];
  d[2] = RS.eq[2 * n + c];
  return true;
}

// pull the 19 post-stream populations of one species: f_i(x) = X_i(x - c_i)
__device__ __forceinline__ void pull19(const double* __restrict__ Xs, const Geom& G, const CellIdx& I, double (&f)[Q]) {
#pragma unroll
  for (int i = 0; i < Q; ++i) f[i] = __ldg(Xs + (long long)i * G.comp + nbr<-1>(I, i));
}

// ---------------------------------------------------------------------------------------------
// two-pass algorithm, pass 1: (rho, phi) of the post-stream populations
// (LBM_hydrovars_density, LBM_binary.H:343-354: sequential sum i = 0..18)
// step_dev / bump: last launch of a CUDA-graph chunk advances the device-side step counter (see k_step_fused)
__global__ void __launch_bounds__(256) k_density(Geom G, const double* __restrict__ X, double2* __restrict__ R,
                                                  long long* step_dev = nullptr, int bump = 0) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zl = blockIdx.z;
  if (step_dev != nullptr && (x | y | zl) == 0) *step_dev += bump;
  if (x >= G.nx || y >= G.ny) return;
  const CellIdx I = cell_idx(G, x, y, zl);
  double f[Q], g[Q];
  pull19(X, G, I, f);
  pull19(X + (long long)Q * G.comp, G, I, g);
  double rho = 0., phi = 0.;
#pragma unroll
  for (int i = 0; i < Q; ++i) { rho += f[i]; phi += g[i]; }
  R[I.zpl[1] + I.yrow[1] + x] = make_double2(rho, phi);
}

// gradients of rho and phi from the density field (LBM_binary.H:134-150)
__device__ __forceinline__ void density_gradients(const double2* __restrict__ R, const CellIdx& I, double (&grho)[3], double (&gphi)[3]) {
  double nr[Q], np[Q];
  nr[0] = np[0] = 0.;
#pragma unroll
  for (int i = 1; i < Q; ++i) {
    const double2 v = __ldg(R + nbr<+1>(I, i));
    nr[i] = v.x;
    np[i] = v.y;
  }
  gradient19(nr, grho);
  gradient19(np, gphi);
}

// two-pass algorithm, pass 2: pull-stream + hydro + collide (+noise) + store.
// Covers K1 (collide_stream, LBM_binary.H:565-573), K4 (thermal_noise :91-128) and K5 (hydrovars :309-311)
// of SURVEY.md 2b in one kernel; the reference's two Swaps (:579-580) become a pointer swap on the host.
// RATE1 (tau_f = tau_g = 1/2): the old populations do not enter the result, the 76 registers that hold them are free after
// the conserved moments are formed.  Two CTAs per SM (<= 128 registers): these kernels serve the small, latency-bound boxes.
template <bool NOISE, bool RATE1>
__global__ void __launch_bounds__(256, RATE1 ? 2 : 1) k_step_twopass(Geom G, DevParams P, long long step_arg, const long long* __restrict__ step_dev,
                                                       const double* __restrict__ X, double* __restrict__ Xn, const double2* __restrict__ R,
                                                       RefState RS) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zl = blockIdx.z;
  if (x >= G.nx || y >= G.ny) return;
  const long long step = step_arg + ((NOISE && step_dev != nullptr) ? *step_dev : 0ll);
  const CellIdx I = cell_idx(G, x, y, zl);
  double f[Q], g[Q], mf[Q], mg[Q];
  pull19(X, G, I, f);
  moments(f, mf);
  pull19(X + (long long)Q * G.comp, G, I, g);
  moments(g, mg);
  double grho[3], gphi[3];
  density_gradients(R, I, grho, gphi);
  const NoiseKey nk = make_noise_key(P.keys, (unsigned long long)cell_global(G, x, y, zl), step);
  CollideCtx C;
  float y3[3], yb[15];
  momentum_normals<NOISE>(nk, y3);
  double ref3[3];
  const bool use_ref = NOISE && ref_densities(G, RS, x, y, zl, ref3);
  collide_prepare<NOISE>(P, grho, gphi, y3, mf, mg, C, use_ref ? ref3 : nullptr);
  const long long c = I.zpl[1] + I.yrow[1] + x;
  double p[Q];
  mode_normals<NOISE, 0>(nk, yb);
  collide_species<NOISE, 0, RATE1>(P, yb, C, mf);
  populations(mf, p);
  const double kf = keep_of(P, 0), kg = keep_of(P, 1);
#pragma unroll
  for (int i = 0; i < Q; ++i) Xn[(long long)i * G.comp + c] = RATE1 ? p[i] : fma(kf, f[i], p[i]);
  mode_normals<NOISE, 1>(nk, yb);
  collide_species<NOISE, 1, RATE1>(P, yb, C, mg);
  populations(mg, p);
#pragma unroll
  for (int i = 0; i < Q; ++i) Xn[(long long)(Q + i) * G.comp + c] = RATE1 ? p[i] : fma(kg, g[i], p[i]);
}

// ---------------------------------------------------------------------------------------------
// plane copies (ghost-plane wrap of a whole-box lattice, halo pack/unpack of a slab)
struct CopyList {
  int n;
  long long src[44], dst[44];  // offsets in doubles
};
// (src and dst may be the same array -- ghost-plane wrap inside one lattice -- so no __restrict__ here)
__global__ void k_copy_planes(CopyList L, const double* src, double* dst, long long count) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int j = blockIdx.y;
  dst[L.dst[j] + i] = src[L.src[j] + i];
}

// ---------------------------------------------------------------------------------------------
// initial conditions.  X_i(x) = w_i * dens(x + c_i), so that the pulled populations are w_i * dens(x)
// like the reference's f(x,y,z,i) = w[i]*rho.
// mode 0 mixture (LBM_binary.H:606-618), 1 stripe (:672-686), 2 droplet (:709-737)
struct InitSpec {
  int mode;
  double rho_lo, rho_hi, kappa, frac, radius;
};
__device__ __forceinline__ void init_density(const InitSpec& S, const Geom& G, int x, int y, int zg, double& rho, double& phi) {
  if (S.mode == 0) {
    rho = 2. * 0.5;
    phi = 2. * 0.5;
  } else if (S.mode == 1) {
    const double pos_lo = (-0.5 * S.frac) * G.nz_global, pos_hi = (0.5 * S.frac) * G.nz_global;
    const double pos = (double)(zg - G.nz_global / 2);  // integer division, LBM_binary.H:680
    const double sk = sqrt(S.kappa);
    rho = (S.rho_hi - S.rho_lo) * 0.5 * (tanh((pos - pos_lo) / sk) + tanh((pos_hi - pos) / sk)) + S.rho_lo;
    phi = (S.rho_hi + S.rho_lo) - rho;
  } else {
    const double Rr = S.radius * G.nx;
    const double rx = x - G.nx / 2., ry = y - G.ny / 2.;
    const double rz = (double)(zg - G.nx / 2);  // box[0] and integer division, LBM_binary.H:725
    const double r = sqrt(rx * rx + ry * ry + rz * rz);
    rho = (S.rho_hi - S.rho_lo) * (1. + tanh((Rr - r) / sqrt(S.kappa))) / 2. + S.rho_lo;
    phi = (S.rho_hi + S.rho_lo) - rho;
  }
}
// fills planes zl = -1 .. nzl (ghost planes included: no exchange needed after an analytic init)
__global__ void __launch_bounds__(256) k_init(Geom G, InitSpec S, double* __restrict__ X, double2* __restrict__ R) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zl = (int)blockIdx.z - 1;
  if (x >= G.nx || y >= G.ny) return;
  const long long c = (long long)(zl + 1) * G.plane + (long long)y * G.nx + x;
  const int nzg = G.nz_global;
#pragma unroll
  for (int i = 0; i < Q; ++i) {
    int xx = x + cx(i), yy = y + cy(i), zz = G.z0 + zl + cz(i);
    xx = xx < 0 ? xx + G.nx : (xx >= G.nx ? xx - G.nx : xx);
    yy = yy < 0 ? yy + G.ny : (yy >= G.ny ? yy - G.ny : yy);
    zz = ((zz % nzg) + nzg) % nzg;
    double rho, phi;
    init_density(S, G, xx, yy, zz, rho, phi);
    X[(long long)i * G.comp + c] = wq(i) * rho;
    X[(long long)(Q + i) * G.comp + c] = wq(i) * phi;
  }
  // densities of the pulled populations, reference order (sum_i w_i * dens)
  {
    const int zg = (((G.z0 + zl) % nzg) + nzg) % nzg;
    double rho, phi, sr = 0., sp = 0.;
    init_density(S, G, x, y, zg, rho, phi);
#pragma unroll
    for (int i = 0; i < Q; ++i) { sr += wq(i) * rho; sp += wq(i) * phi; }
    R[c] = make_double2(sr, sp);
  }
}

// Restart upload (LBM_init, LBM_binary.H:631-661): the host holds post-stream populations f_i(x); the lattice stores
// them pre-stream, X_i(x - c_i) = f_i(x).  PUSH formulation: the chunk of host planes [zs, zs + gridDim.z) that has
// just landed in `stage` (component-major, exactly those planes, no ghost planes) is written to its targets; every
// lattice entry has exactly one source, so chunks are independent and nothing is uploaded twice.
// wrap_z: whole box (targets wrap periodically); otherwise targets outside the slab belong to the neighbour and are
// dropped (the host array of a slab carries the two ghost planes zs = -1 and nzl as sources for that reason).
__global__ void __launch_bounds__(256) k_scatter_populations(Geom G, int zs0, int wrap_z, const double* __restrict__ stage,
                                                              double* __restrict__ X) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zs = zs0 + (int)blockIdx.z;
  if (x >= G.nx || y >= G.ny) return;
  const int xs[3] = {x == 0 ? G.nx - 1 : x - 1, x, x == G.nx - 1 ? 0 : x + 1};
  const long long yr[3] = {(long long)(y == 0 ? G.ny - 1 : y - 1) * G.nx, (long long)y * G.nx, (long long)(y == G.ny - 1 ? 0 : y + 1) * G.nx};
  const long long scomp = (long long)gridDim.z * G.plane;
  const long long s = (long long)blockIdx.z * G.plane + yr[1] + x;
#pragma unroll
  for (int i = 0; i < Q; ++i) {
    int zt = zs - cz(i);
    if (wrap_z) zt = zt < 0 ? zt + G.nzl : (zt >= G.nzl ? zt - G.nzl : zt);
    if (zt < 0 || zt >= G.nzl) continue;
    const long long t = (long long)(zt + 1) * G.plane + yr[1 - cy(i)] + xs[1 - cx(i)];
    X[(long long)i * G.comp + t] = stage[(long long)i * scomp + s];
    X[(long long)(Q + i) * G.comp + t] = stage[(long long)(Q + i) * scomp + s];
  }
}

// ---------------------------------------------------------------------------------------------
// observers: everything the reference keeps in hydrovs / hydrovsbar / fnoisevs / gnoisevs / fold / gold is
// recomputed on demand from (X, R) for planes [zlo, zlo + gridDim.z).  out is component-major over the chunk.
enum ObserveMode { OBS_POP = 0, OBS_HYDRO = 1, OBS_HBAR = 2, OBS_NOISE = 3, OBS_NORMALS = 4 };

template <int MODE, bool NOISE>
__global__ void __launch_bounds__(256) k_observe(Geom G, DevParams P, long long step, int zlo, const double* __restrict__ X,
                                                  const double2* __restrict__ R, double* __restrict__ out, RefState RS) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zc = blockIdx.z, zl = zlo + zc;
  if (x >= G.nx || y >= G.ny) return;
  const CellIdx I = cell_idx(G, x, y, zl);
  const long long oc = (long long)gridDim.z * G.plane;                       // component stride of the chunk
  const long long o = (long long)zc * G.plane + (long long)y * G.nx + x;    // cell offset in the chunk
  const NoiseKey nk = make_noise_key(P.keys, (unsigned long long)cell_global(G, x, y, zl), step);
  if (MODE == OBS_NORMALS) {
    float n[36];
    cell_normals(nk, n);
#pragma unroll
    for (int d = 0; d < 33; ++d) out[o * 33 + d] = normal_of(n[d]);
    return;
  }
  double f[Q], g[Q];
  pull19(X, G, I, f);
  pull19(X + (long long)Q * G.comp, G, I, g);
  if (MODE == OBS_POP) {
#pragma unroll
    for (int i = 0; i < Q; ++i) { out[(long long)i * oc + o] = f[i]; out[(long long)(Q + i) * oc + o] = g[i]; }
    return;
  }
  double mf[Q], mg[Q];
  moments(f, mf);
  moments(g, mg);
  // rho, phi as the reference's hydrovars_bar_density: sequential sums (LBM_binary.H:322-330)
  double rho = 0., phi = 0.;
#pragma unroll
  for (int i = 0; i < Q; ++i) { rho += f[i]; phi += g[i]; }
  if (MODE == OBS_HBAR) {
    const bool hf = fabs(mf[0]) > (double)FLT_EPSILON, hg = fabs(mg[0]) > (double)FLT_EPSILON;
    out[0 * oc + o] = rho;
    out[1 * oc + o] = phi;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      out[(2 + k) * oc + o] = hf ? mf[1 + k] / mf[0] : 0.;
      out[(6 + k) * oc + o] = hg ? mg[1 + k] / mg[0] : 0.;
    }
    out[5 * oc + o] = mf[0] + mg[0];
    return;
  }
  float n[36];
  if (NOISE) cell_normals(nk, n);
  else {
#pragma unroll
    for (int d = 0; d < 36; ++d) n[d] = NRM_BIAS_F;
  }
  double ref3[3] = {rho, phi, rho + phi};
  const bool use_ref = NOISE && ref_densities(G, RS, x, y, zl, ref3);
  if (MODE == OBS_NOISE) {
    // fnoisevs / gnoisevs (LBM_binary.H:113-127; amplitudes from the reference state under USE_REF_STATE, :92-107)
    const double aj = NOISE ? sqrt(P.amp_j * fabs(ref3[0] * ref3[1] / ref3[2])) : 0.;
    const double sf = NOISE ? sqrt(P.amp_s * fabs(ref3[0])) : 0., sg = NOISE ? sqrt(P.amp_s * fabs(ref3[1])) : 0.;
    out[0 * oc + o] = 0.;
    out[(long long)Q * oc + o] = 0.;
#pragma unroll
    for (int a = 1; a <= 3; ++a) {
      const double v = aj * normal_of(n[a - 1]);
      out[(long long)a * oc + o] = v;
      out[(long long)(Q + a) * oc + o] = -v;
    }
#pragma unroll
    for (int a = 4; a < Q; ++a) {
      out[(long long)a * oc + o] = (sqrt_bnorm(a) * sf) * normal_of(n[3 + 2 * (a - 4)]);
      out[(long long)(Q + a) * oc + o] = (sqrt_bnorm(a) * sg) * normal_of(n[4 + 2 * (a - 4)]);
    }
    return;
  }
  if (MODE == OBS_HYDRO) {
    double grho[3], gphi[3];
    density_gradients(R, I, grho, gphi);
    const float n3[3] = {n[0], n[1], n[2]};
    const double jf[3] = {mf[1], mf[2], mf[3]}, jg[3] = {mg[1], mg[2], mg[3]};
    CellHydro H;
    double sq_rho, sq_phi;
    cell_hydro<NOISE>(P, rho, phi, jf, jg, grho, gphi, n3, H, sq_rho, sq_phi, use_ref ? ref3 : nullptr);
    out[0 * oc + o] = rho;
    out[1 * oc + o] = phi;
    out[5 * oc + o] = rho + phi;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      out[(2 + k) * oc + o] = H.uf[k];
      out[(6 + k) * oc + o] = H.ug[k];
      out[(9 + k) * oc + o] = H.af[k];
      out[(12 + k) * oc + o] = H.ag[k];
      out[(15 + k) * oc + o] = (rho * H.ufb[k] + phi * H.ugb[k] + 0.5 * (rho * H.af[k] + phi * H.ag[k])) * H.inv_tot;
    }
    out[18 * oc + o] = H.nfv[0];
    out[19 * oc + o] = H.ngv[0];
    out[20 * oc + o] = H.ufb[0];
    out[21 * oc + o] = H.ugb[0];
  }
}

// diagnostics: per-block partial sums {rho, phi, rho*x, rho*y, rho*zg, rho*xx, rho*yy, rho*zz, rho*xy, rho*xz, rho*yz}
// (cell indices as coordinates; zg = global plane) and count of non-finite densities.  First moments: update_com
// (LBM_hydrovs.H:26-60); second moments: the mass-weighted covariance of fittingDropletCovariance (LBM_hydrovs.H:258-335).
constexpr int NDIAG = 11;
__global__ void __launch_bounds__(256) k_diag(Geom G, const double2* __restrict__ R, double* __restrict__ partial,
                                               unsigned long long* __restrict__ nonfinite) {
  __shared__ double sh[NDIAG][256];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zl = blockIdx.z;
  double v[NDIAG];
#pragma unroll
  for (int k = 0; k < NDIAG; ++k) v[k] = 0.;
  if (x < G.nx && y < G.ny) {
    const double2 r = R[(long long)(zl + 1) * G.plane + (long long)y * G.nx + x];
    const double X = x, Y = y, Z = G.z0 + zl;
    v[0] = r.x; v[1] = r.y; v[2] = r.x * X; v[3] = r.x * Y; v[4] = r.x * Z;
    v[5] = v[2] * X; v[6] = v[3] * Y; v[7] = v[4] * Z; v[8] = v[2] * Y; v[9] = v[2] * Z; v[10] = v[3] * Z;
    if (!(isfinite(r.x) && isfinite(r.y))) atomicAdd(nonfinite, 1ull);
  }
#pragma unroll
  for (int k = 0; k < NDIAG; ++k) sh[k][tid] = v[k];
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (tid < s) {
#pragma unroll
      for (int k = 0; k < NDIAG; ++k) sh[k][tid] += sh[k][tid + s];
    }
    __syncthreads();
  }
  if (tid == 0) {
    const long long b = ((long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
#pragma unroll
    for (int k = 0; k < NDIAG; ++k) partial[b * NDIAG + k] = sh[k][0];
  }
}
// Field terms of the droplet (W, R) fit (externlib.H:246-340: func_MfWn_mult, func_MfRn_mult): per-block partial sums of
//   rho (R - r') sech^2((R - r') / s)   and   rho sech^2((R - r') / s),   r' = |r - r0|, unit-cube cell-centre coordinates,
// plus (MINMAX) the block's min / max of rho for C0 = max rho - min rho (LBM_hydrovs.H:124-125).  partial: [block][4].
__global__ void __launch_bounds__(256) k_fit_terms(Geom G, const double2* __restrict__ R, double inv_s, double Rn, double r0x, double r0y,
                                                    double r0z, double* __restrict__ partial) {
  __shared__ double sh[4][256];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zl = blockIdx.z;
  double v0 = 0., v1 = 0., mn = 1e300, mx = -1e300;
  if (x < G.nx && y < G.ny) {
    const double rho = R[(long long)(zl + 1) * G.plane + (long long)y * G.nx + x].x;
    const double dx = (x + 0.5) / G.nx - r0x, dy = (y + 0.5) / G.ny - r0y, dz = (G.z0 + zl + 0.5) / G.nz_global - r0z;
    const double dist = Rn - sqrt(dx * dx + dy * dy + dz * dz), a = dist * inv_s;
    const double sech = fabs(a) < 710.4 ? 1. / cosh(a) : 0.;  // inv_acosh, externlib.H:23-30
    v1 = rho * (sech * sech);
    v0 = rho * (dist * sech * sech);
    mn = mx = rho;
  }
  sh[0][tid] = v0; sh[1][tid] = v1; sh[2][tid] = mn; sh[3][tid] = mx;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (tid < s) {
      sh[0][tid] += sh[0][tid + s];
      sh[1][tid] += sh[1][tid + s];
      sh[2][tid] = fmin(sh[2][tid], sh[2][tid + s]);
      sh[3][tid] = fmax(sh[3][tid], sh[3][tid + s]);
    }
    __syncthreads();
  }
  if (tid == 0) {
    const long long b = ((long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) partial[b * 4 + k] = sh[k][0];
  }
}

// update_com for the reference-state noise (LBM_hydrovs.H:26-60, LBM_binary.H:586-588): block partials of k_diag summed in block
// order by one thread block (deterministic), shift = (int)(com - com_ref) per axis (C truncation, like the reference's static_cast)
__global__ void __launch_bounds__(256) k_com_shift(const double* __restrict__ partial, long long nblocks, double cx, double cy, double cz,
                                                    int* __restrict__ shift) {
  __shared__ double sh[4][256];
  double v[4] = {0., 0., 0., 0.};
  const int pick[4] = {0, 2, 3, 4};
  // thread t sums blocks t, t + 256, ... in order; then a fixed tree
  for (long long b = threadIdx.x; b < nblocks; b += 256)
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] += partial[b * NDIAG + pick[k]];
#pragma unroll
  for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] = v[k];
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) {
#pragma unroll
      for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double m = sh[0][0];
    shift[0] = (int)(sh[1][0] / m - cx);
    shift[1] = (int)(sh[2][0] / m - cy);
    shift[2] = (int)(sh[3][0] / m - cz);
  }
}
// Centre of mass of the brick kernels (reference-state noise on a whole box or a slab): com[4 zg .. 4 zg + 3] = {sum rho, sum rho x,
// sum rho y, sum rho zg} of every GLOBAL plane zg over R (cell indices as coordinates, like k_diag).  Two levels in a fixed order
// that depends on (nx, ny) only -- not on the brick grid, the slab cut or the schedule:
//   k_com_chunks : CTA (chunk, zl) sums the COM_CHUNK cells [chunk * COM_CHUNK, ...) of plane zl, thread t the cells t, t + 256, ...
//                  of the chunk in order, then a fixed tree -> part[zl][chunk][4]  (many CTAs even for a thin slab of large planes)
//   k_com_fold_chunks : one thread per global plane adds its chunks in order; planes outside this slab get zeros, so that a sum
//                  all-reduce of the buffers of all slabs is exact (one contributor per entry) and completes every slab's copy.
constexpr int COM_THREADS = 256, COM_CHUNK = 32 * COM_THREADS;
inline int com_chunks(const Geom& G) { return (int)((G.plane + COM_CHUNK - 1) / COM_CHUNK); }
__global__ void __launch_bounds__(COM_THREADS) k_com_chunks(Geom G, const double2* __restrict__ R, double* __restrict__ part) {
  __shared__ double sh[4][COM_THREADS];
  const int zl = blockIdx.y, t = threadIdx.x, c0 = blockIdx.x * COM_CHUNK;
  const int c1 = (int)min((long long)c0 + COM_CHUNK, G.plane);  // a plane is < 2^29 cells (4 GiB per component, create_common)
  const double2* Rp = R + (long long)(zl + 1) * G.plane;
  const double Z = G.z0 + zl;
  double v[4] = {0., 0., 0., 0.};
#pragma unroll 8
  for (int c = c0 + t; c < c1; c += COM_THREADS) {
    const int y = c / G.nx, x = c - y * G.nx;
    const double r = __ldg(&Rp[c].x);
    v[0] += r; v[1] += r * (double)x; v[2] += r * (double)y; v[3] += r * Z;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) sh[k][t] = v[k];
  __syncthreads();
  for (int s = COM_THREADS / 2; s > 0; s >>= 1) {
    if (t < s) {
#pragma unroll
      for (int k = 0; k < 4; ++k) sh[k][t] += sh[k][t + s];
    }
    __syncthreads();
  }
  if (t < 4) part[((long long)zl * gridDim.x + blockIdx.x) * 4 + t] = sh[t][0];
}
__global__ void k_com_fold_chunks(Geom G, const double* __restrict__ part, int nchunk, double* __restrict__ com) {
  const int zg = blockIdx.x * blockDim.x + threadIdx.x, zl = zg - G.z0;
  if (zg >= G.nz_global) return;
  double v[4] = {0., 0., 0., 0.};
  if (zl >= 0 && zl < G.nzl)
    for (int j = 0; j < nchunk; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] += part[((long long)zl * nchunk + j) * 4 + k];
#pragma unroll
  for (int k = 0; k < 4; ++k) com[4ll * zg + k] = v[k];
}
// sums the nz plane vectors of k_com_fold_chunks in z order (one thread: the same bits on every slab of a box) and writes
// shift = (int)(com - c) per axis (C truncation, like the reference's static_cast)
__global__ void k_com_shift_planes(const double* __restrict__ com, int nz, double cx, double cy, double cz, int* __restrict__ shift) {
  double s[4] = {0., 0., 0., 0.};
  for (int z = 0; z < nz; ++z)
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] += com[4ll * z + k];
  shift[0] = (int)(s[1] / s[0] - cx);
  shift[1] = (int)(s[2] / s[0] - cy);
  shift[2] = (int)(s[3] / s[0] - cz);
}
__global__ void k_count_nonfinite(const double* __restrict__ a, long long n, unsigned long long* __restrict__ cnt) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !isfinite(a[i])) atomicAdd(cnt, 1ull);
}

__global__ void k_philox_test(uint4 ctr, uint2 key, uint4* out) { *out = philox4x32(ctr, key); }

// Deep statistics of the in-kernel Gaussian generator (test hook): the 33 normals of `ncells` cells over `nsteps` steps, i.e. exactly
// what the step kernels would draw, binned on the device.  hist: nbins equal bins over [lo, hi) + underflow + overflow, all 33
// streams pooled; joint: JB x JB bins over [-4, 4)^2 of the two normals that come out of ONE Philox word (cos / sin branch of a
// Box-Muller pair; draws (0,1), (2,3) ... of species f), the place where a dependence would show; mom: sums of n, n^2, n^3, n^4.
constexpr int NORMAL_JOINT_BINS = 32;
__global__ void __launch_bounds__(256) k_normal_stats(PhiloxKeys K, long long ncells, long long step0, int nsteps, int nbins, double lo, double hi,
                                                       unsigned long long* __restrict__ hist, unsigned long long* __restrict__ joint,
                                                       double* __restrict__ mom) {
  extern __shared__ unsigned int sh[];  // [nbins + 2] + [JB * JB]
  unsigned int* sj = sh + nbins + 2;
  const int nsh = nbins + 2 + NORMAL_JOINT_BINS * NORMAL_JOINT_BINS;
  for (int i = threadIdx.x; i < nsh; i += blockDim.x) sh[i] = 0u;
  __syncthreads();
  const double inv_w = nbins / (hi - lo);
  double m1 = 0., m2 = 0., m3 = 0., m4 = 0.;
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
    for (int s = 0; s < nsteps; ++s) {
      const NoiseKey nk = make_noise_key(K, (unsigned long long)c, step0 + s);
      float F[19], G[16];
      species_normals<0, 0, 18>(nk, F);
      species_normals<1, 0, 15>(nk, G);
#pragma unroll
      for (int j = 0; j < 33; ++j) {
        const double n = normal_of(j < 18 ? F[j] : G[j - 18]);
        const double b = floor((n - lo) * inv_w);
        const int bin = b < 0. ? nbins : (b >= nbins ? nbins + 1 : (int)b);
        atomicAdd(&sh[bin], 1u);
        const double n2 = n * n;
        m1 += n; m2 += n2; m3 += n2 * n; m4 += n2 * n2;
      }
#pragma unroll
      for (int j = 0; j < 18; j += 2) {
        const double a = normal_of(F[j]), b = normal_of(F[j + 1]);
        const int ia = (int)floor((a + 4.) * (NORMAL_JOINT_BINS / 8.)), ib = (int)floor((b + 4.) * (NORMAL_JOINT_BINS / 8.));
        if (ia >= 0 && ia < NORMAL_JOINT_BINS && ib >= 0 && ib < NORMAL_JOINT_BINS) atomicAdd(&sj[ia * NORMAL_JOINT_BINS + ib], 1u);
      }
    }
    // flush often enough that the 32-bit shared counters cannot overflow (<= 33 * nsteps per cell and thread)
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nbins + 2; i += blockDim.x) if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
  for (int i = threadIdx.x; i < NORMAL_JOINT_BINS * NORMAL_JOINT_BINS; i += blockDim.x) if (sj[i]) atomicAdd(&joint[i], (unsigned long long)sj[i]);
  atomicAdd(&mom[0], m1); atomicAdd(&mom[1], m2); atomicAdd(&mom[2], m3); atomicAdd(&mom[3], m4);
}

}  // namespace bflbm
