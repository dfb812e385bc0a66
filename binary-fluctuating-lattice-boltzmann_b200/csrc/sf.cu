// On-GPU structure-factor accumulator (include/bflbm_sf.h): hydrovs on the device -> cuFFT D2Z per distinct variable
// -> running sums of A_k conj(B_k) per pair.  Built as its own library on top of libbflbm.so's public C ABI.
#include <vector>

#include "../../include/bflbm_sf.h"
#include "sf_common.cuh"

namespace {
// one pair: half spectrum -> full shifted grid (Hermitian completion: S(-k) = conj S(k)), mean over samples, k = 0 bin
__global__ void k_sf_expand(int nx, int ny, int nz, int nxh, const double* __restrict__ acc_re, const double* __restrict__ acc_im,
                            double inv_samples, int zero_avg, double* __restrict__ out_re, double* __restrict__ out_im) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
  if (x >= nx) return;
  // shifted index -> frequency index (fftshift moves frequency 0 to n/2)
  const int kx = (x + nx - nx / 2) % nx, ky = (y + ny - ny / 2) % ny, kz = (z + nz - nz / 2) % nz;
  double re, im;
  if (kx < nxh) {
    const long long i = ((long long)kz * ny + ky) * nxh + kx;
    re = acc_re[i];
    im = acc_im[i];
  } else {
    const long long i = ((long long)((nz - kz) % nz) * ny + (ny - ky) % ny) * nxh + (nx - kx);
    re = acc_re[i];
    im = -acc_im[i];
  }
  if (zero_avg && kx == 0 && ky == 0 && kz == 0) re = im = 0.;
  const long long o = ((long long)z * ny + y) * nx + x;
  out_re[o] = re * inv_samples;
  if (out_im) out_im[o] = im * inv_samples;
}
}  // namespace

struct bflbm_sf {
  std::vector<bflbm_lattice*> lats;  // the whole-box lattice, or every slab of a box (bflbm_sf_create_multi)
  int device = 0;                    // where the assembled fields, the FFTs and the running sums live (the first lattice's GPU)
  int nx = 0, ny = 0, nz = 0, nxh = 0, npairs = 0, nvars = 0;
  long long n = 0, nhalf = 0, samples = 0;
  std::vector<int> vars;  // distinct hydrovs components, in order of first use
  cufftHandle plan = 0;
  bool have_plan = false;
  double* hydro = nullptr;              // [22][n]
  cufftDoubleComplex* spec = nullptr;   // [nvars][nhalf]
  double *acc_re = nullptr, *acc_im = nullptr, *scale = nullptr, *full = nullptr;  // [npairs][nhalf] x2, [npairs], [2][n]
  int *slotA = nullptr, *slotB = nullptr;
};

extern "C" {

static int sf_create_common(const std::vector<bflbm_lattice*>& lats, int npairs, const int* pairA, const int* pairB, const double* var_scaling,
                            bflbm_sf** out) {
  if (lats.empty() || !lats[0] || !out || npairs < 1 || !pairA || !pairB) return sf_fail(BFLBM_ERR_ARG, "bad argument");
  *out = nullptr;
  int nx, ny, nz, z0, nzg;
  if (bflbm_get_dims(lats[0], &nx, &ny, &nz, &z0, &nzg)) return sf_fail(BFLBM_ERR_ARG, "cannot query the lattice");
  long long covered = 0;
  for (bflbm_lattice* l : lats) {
    int lx, ly, lz, l0, lg;
    if (!l || bflbm_get_dims(l, &lx, &ly, &lz, &l0, &lg) || lx != nx || ly != ny || lg != nzg) return sf_fail(BFLBM_ERR_ARG, "lattices of different boxes");
    covered += lz;
  }
  if (covered != nzg) return sf_fail(BFLBM_ERR_ARG, "structure factors need the whole box: one whole-box lattice, or all slabs (bflbm_sf_create_multi)");
  nz = nzg;
  bflbm_sf* s = new bflbm_sf;
  s->lats = lats;
  s->device = bflbm_get_device(lats[0]);
  SF_CU(cudaSetDevice(s->device));
  s->nx = nx; s->ny = ny; s->nz = nz; s->nxh = nx / 2 + 1; s->npairs = npairs;
  s->n = (long long)nx * ny * nz;
  s->nhalf = (long long)s->nxh * ny * nz;
  std::vector<int> sa(npairs), sb(npairs);
  std::vector<double> sc(npairs, 1.0);
  auto slot = [&](int v) {
    for (size_t i = 0; i < s->vars.size(); ++i) if (s->vars[i] == v) return (int)i;
    s->vars.push_back(v);
    return (int)s->vars.size() - 1;
  };
  for (int p = 0; p < npairs; ++p) {
    if (pairA[p] < 0 || pairA[p] >= BFLBM_NHYDRO || pairB[p] < 0 || pairB[p] >= BFLBM_NHYDRO) {
      delete s;
      return sf_fail(BFLBM_ERR_ARG, "pair index outside hydrovs (0..21)");
    }
    sa[p] = slot(pairA[p]);
    sb[p] = slot(pairB[p]);
    if (var_scaling) sc[p] = var_scaling[p];
  }
  s->nvars = (int)s->vars.size();
#define SF_TRY(x) do { int rc_ = (x); if (rc_) { bflbm_sf_destroy(s); return rc_; } } while (0)
  auto alloc = [&](void** p, size_t bytes) -> int { SF_CU(cudaMalloc(p, bytes)); return 0; };
  SF_TRY(alloc((void**)&s->hydro, (size_t)BFLBM_NHYDRO * s->n * sizeof(double)));
  SF_TRY(alloc((void**)&s->spec, (size_t)s->nvars * s->nhalf * sizeof(cufftDoubleComplex)));
  SF_TRY(alloc((void**)&s->acc_re, (size_t)npairs * s->nhalf * sizeof(double)));
  SF_TRY(alloc((void**)&s->acc_im, (size_t)npairs * s->nhalf * sizeof(double)));
  SF_TRY(alloc((void**)&s->full, (size_t)2 * s->n * sizeof(double)));
  SF_TRY(alloc((void**)&s->scale, npairs * sizeof(double)));
  SF_TRY(alloc((void**)&s->slotA, npairs * sizeof(int)));
  SF_TRY(alloc((void**)&s->slotB, npairs * sizeof(int)));
  cudaMemcpy(s->scale, sc.data(), npairs * sizeof(double), cudaMemcpyHostToDevice);
  cudaMemcpy(s->slotA, sa.data(), npairs * sizeof(int), cudaMemcpyHostToDevice);
  cudaMemcpy(s->slotB, sb.data(), npairs * sizeof(int), cudaMemcpyHostToDevice);
  if (cufftPlan3d(&s->plan, nz, ny, nx, CUFFT_D2Z) != CUFFT_SUCCESS) { bflbm_sf_destroy(s); return sf_fail(BFLBM_ERR_CUDA, "cufftPlan3d failed"); }
  s->have_plan = true;
  SF_TRY(bflbm_sf_reset(s));
#undef SF_TRY
  *out = s;
  return 0;
}

int bflbm_sf_create(bflbm_lattice* h, int npairs, const int* pairA, const int* pairB, const double* var_scaling, bflbm_sf** out) {
  return sf_create_common(std::vector<bflbm_lattice*>{h}, npairs, pairA, pairB, var_scaling, out);
}
int bflbm_sf_create_multi(bflbm_multi* m, int npairs, const int* pairA, const int* pairB, const double* var_scaling, bflbm_sf** out) {
  std::vector<bflbm_lattice*> lats;
  for (int i = 0; i < bflbm_multi_count(m); ++i) lats.push_back(bflbm_multi_slab(m, i));
  return sf_create_common(lats, npairs, pairA, pairB, var_scaling, out);
}

int bflbm_sf_destroy(bflbm_sf* s) {
  if (!s) return 0;
  cudaSetDevice(s->device);
  if (s->have_plan) cufftDestroy(s->plan);
  cudaFree(s->hydro); cudaFree(s->spec); cudaFree(s->acc_re); cudaFree(s->acc_im); cudaFree(s->full);
  cudaFree(s->scale); cudaFree(s->slotA); cudaFree(s->slotB);
  delete s;
  return 0;
}

int bflbm_sf_reset(bflbm_sf* s) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  SF_CU(cudaSetDevice(s->device));
  SF_CU(cudaMemset(s->acc_re, 0, (size_t)s->npairs * s->nhalf * sizeof(double)));
  SF_CU(cudaMemset(s->acc_im, 0, (size_t)s->npairs * s->nhalf * sizeof(double)));
  s->samples = 0;
  return 0;
}

long long bflbm_sf_samples(const bflbm_sf* s) { return s ? s->samples : -1; }

int bflbm_sf_accumulate(bflbm_sf* s) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  // every lattice writes its planes of the 22 fields into the assembled array (a peer copy from the other GPUs' slabs);
  // each call synchronises that lattice's stream
  for (bflbm_lattice* l : s->lats) {
    const int rc = bflbm_get_hydrovars_device_into_global(l, s->hydro);
    if (rc) return sf_fail(rc, bflbm_last_error());
  }
  SF_CU(cudaSetDevice(s->device));
  for (int v = 0; v < s->nvars; ++v)
    if (cufftExecD2Z(s->plan, s->hydro + (long long)s->vars[v] * s->n, s->spec + (long long)v * s->nhalf) != CUFFT_SUCCESS)
      return sf_fail(BFLBM_ERR_CUDA, "cufftExecD2Z failed");
  const int T = 256;
  k_sf_accumulate<<<(unsigned)((s->nhalf + T - 1) / T), T>>>(s->nhalf, s->npairs, s->slotA, s->slotB, s->scale, s->spec, 1.0 / (double)s->n,
                                                             s->acc_re, s->acc_im);
  SF_CU(cudaGetLastError());
  SF_CU(cudaDeviceSynchronize());
  ++s->samples;
  return 0;
}

int bflbm_sf_get(bflbm_sf* s, int zero_avg, double* real, double* imag) {
  if (!s || !real) return sf_fail(BFLBM_ERR_ARG, "null argument");
  if (s->samples == 0) return sf_fail(BFLBM_ERR_STATE, "no samples accumulated");
  SF_CU(cudaSetDevice(s->device));
  const dim3 block(128), grid((s->nx + 127) / 128, s->ny, s->nz);
  for (int p = 0; p < s->npairs; ++p) {
    k_sf_expand<<<grid, block>>>(s->nx, s->ny, s->nz, s->nxh, s->acc_re + (long long)p * s->nhalf, s->acc_im + (long long)p * s->nhalf,
                                 1.0 / (double)s->samples, zero_avg, s->full, imag ? s->full + s->n : nullptr);
    SF_CU(cudaGetLastError());
    SF_CU(cudaMemcpy(real + (long long)p * s->n, s->full, s->n * sizeof(double), cudaMemcpyDeviceToHost));
    if (imag) SF_CU(cudaMemcpy(imag + (long long)p * s->n, s->full + s->n, s->n * sizeof(double), cudaMemcpyDeviceToHost));
  }
  return 0;
}

}  // extern "C"
