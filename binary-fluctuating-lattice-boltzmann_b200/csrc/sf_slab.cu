// Structure factors of a box split over ranks (include/bflbm_sf_slab.h): slab FFT with one all-to-all transpose per variable,
// every rank keeping its slab of the fields and its kx columns of k-space.  The caller moves the all-to-all blocks.
#include <algorithm>
#include <vector>

#include "../../include/bflbm_sf_slab.h"
#include "sf_common.cuh"

namespace {
// the kx columns [0, nxh) split into P contiguous ranges, remainder to the low ranks (like distributed.slab_bounds)
struct KxSplit {
  int base, rem;
  __host__ __device__ int first(int r) const { return r * base + (r < rem ? r : rem); }
  __host__ __device__ int count(int r) const { return base + (r < rem ? 1 : 0); }
  __host__ __device__ int owner(int kx) const {
    const int big = rem * (base + 1);
    return kx < big ? kx / (base + 1) : rem + (kx - big) / base;
  }
};

// [z][ky][kx] of the local planes (rows = nz_local * ny) -> send block of rank d = owner(kx), laid out [z][ky][kx - kx0_d]
__global__ void k_sf_slab_pack(long long rows, int nxh, KxSplit split, const cufftDoubleComplex* __restrict__ in,
                               cufftDoubleComplex* __restrict__ send) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * nxh) return;
  const long long row = i / nxh;
  const int kx = (int)(i - row * nxh);
  const int d = split.owner(kx), kx0 = split.first(d), nkx = split.count(d);
  send[rows * kx0 + row * nkx + (kx - kx0)] = in[i];
}

// One pair: the rank's half-spectrum columns [kx0, kx0 + nkx) (layout [kz][ky][kx - kx0]) -> the shifted x columns it owns,
// compact [z][y][c] with x = colx[c]; Hermitian completion for kx >= nxh, mean over samples, k = 0 bin
__global__ void k_sf_slab_expand(int nx, int ny, int nz, int nxh, int kx0, int nkx, int ncols, const int* __restrict__ colx,
                                 const double* __restrict__ acc_re, const double* __restrict__ acc_im, double inv_samples,
                                 int zero_avg, double* __restrict__ out_re, double* __restrict__ out_im) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
  if (c >= ncols) return;
  const int x = colx[c];
  const int kx = (x + nx - nx / 2) % nx, ky = (y + ny - ny / 2) % ny, kz = (z + nz - nz / 2) % nz;
  double re, im;
  if (kx < nxh) {
    const long long i = ((long long)kz * ny + ky) * nkx + (kx - kx0);
    re = acc_re[i];
    im = acc_im[i];
  } else {
    const long long i = ((long long)((nz - kz) % nz) * ny + (ny - ky) % ny) * nkx + (nx - kx - kx0);
    re = acc_re[i];
    im = -acc_im[i];
  }
  if (zero_avg && kx == 0 && ky == 0 && kz == 0) re = im = 0.;
  const long long o = ((long long)z * ny + y) * ncols + c;
  out_re[o] = re * inv_samples;
  out_im[o] = im * inv_samples;
}
}  // namespace

struct bflbm_sf_slab {
  bflbm_lattice* lat = nullptr;
  int device = 0, nranks = 1, rank = 0;
  std::vector<int> zsplit;
  KxSplit split{};
  int nx = 0, ny = 0, nz = 0, nzl = 0, nxh = 0, kx0 = 0, nkx = 0, npairs = 0, nvars = 0;
  long long n = 0;      // cells of the whole box
  long long n2d = 0;    // complex values of one variable's 2-D transforms: nz_local * ny * nxh
  long long ncol = 0;   // complex values of one variable on this rank's kx columns: nz * ny * nkx
  long long samples = 0;
  int next_round = 0, open_round = -1;
  std::vector<int> vars;  // distinct hydrovs components, in order of first use; round v transforms vars[v]
  std::vector<int> colx;  // shifted x columns this rank writes in get, ascending
  cudaStream_t stream = nullptr;
  cufftHandle plan2d = 0, planz = 0;
  bool have2d = false, havez = false;
  void* work = nullptr;                 // cuFFT work area shared by both plans
  double* hydro = nullptr;              // [22][nz_local][ny][nx]
  cufftDoubleComplex *out2d = nullptr, *send = nullptr, *recv = nullptr;  // n2d, n2d, ncol
  cufftDoubleComplex* spec = nullptr;   // [nvars][ncol]
  double *acc_re = nullptr, *acc_im = nullptr, *scale = nullptr;  // [npairs][ncol] x2, [npairs]
  int *slotA = nullptr, *slotB = nullptr, *d_colx = nullptr;
};

extern "C" {

int bflbm_sf_slab_destroy(bflbm_sf_slab* s) {
  if (!s) return 0;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  if (s->have2d) cufftDestroy(s->plan2d);
  if (s->havez) cufftDestroy(s->planz);
  cudaFree(s->work); cudaFree(s->hydro); cudaFree(s->out2d); cudaFree(s->send); cudaFree(s->recv); cudaFree(s->spec);
  cudaFree(s->acc_re); cudaFree(s->acc_im); cudaFree(s->scale); cudaFree(s->slotA); cudaFree(s->slotB); cudaFree(s->d_colx);
  delete s;
  return 0;
}

int bflbm_sf_slab_reset(bflbm_sf_slab* s) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  SF_CU(cudaSetDevice(s->device));
  SF_CU(cudaMemsetAsync(s->acc_re, 0, (size_t)s->npairs * s->ncol * sizeof(double), s->stream));
  SF_CU(cudaMemsetAsync(s->acc_im, 0, (size_t)s->npairs * s->ncol * sizeof(double), s->stream));
  s->samples = 0;
  s->next_round = 0;
  s->open_round = -1;
  return 0;
}

int bflbm_sf_slab_create(bflbm_lattice* lat, int nranks, int rank, const int* zsplit, int npairs, const int* pairA,
                         const int* pairB, const double* var_scaling, bflbm_sf_slab** out) {
  if (!out) return sf_fail(BFLBM_ERR_ARG, "null output handle");
  *out = nullptr;
  if (!lat || nranks < 1 || rank < 0 || rank >= nranks || !zsplit || npairs < 1 || !pairA || !pairB)
    return sf_fail(BFLBM_ERR_ARG, "bad argument");
  int nx, ny, nzl, z0, nz;
  if (bflbm_get_dims(lat, &nx, &ny, &nzl, &z0, &nz)) return sf_fail(BFLBM_ERR_ARG, "cannot query the lattice");
  if (zsplit[0] != 0 || zsplit[nranks] != nz) return sf_fail(BFLBM_ERR_ARG, "zsplit must run from 0 to nz");
  for (int r = 0; r < nranks; ++r)
    if (zsplit[r + 1] <= zsplit[r]) return sf_fail(BFLBM_ERR_ARG, "zsplit must be strictly increasing");
  if (zsplit[rank] != z0 || zsplit[rank + 1] - zsplit[rank] != nzl)
    return sf_fail(BFLBM_ERR_ARG, "the lattice's planes are not [zsplit[rank], zsplit[rank + 1])");
  const int nxh = nx / 2 + 1;
  if (nxh < nranks) return sf_fail(BFLBM_ERR_ARG, "nx/2 + 1 < nranks: some rank would own no kx column");
  for (int p = 0; p < npairs; ++p)
    if (pairA[p] < 0 || pairA[p] >= BFLBM_NHYDRO || pairB[p] < 0 || pairB[p] >= BFLBM_NHYDRO)
      return sf_fail(BFLBM_ERR_ARG, "pair index outside hydrovs (0..21)");

  bflbm_sf_slab* s = new bflbm_sf_slab;
  s->lat = lat;
  s->device = bflbm_get_device(lat);
  s->nranks = nranks;
  s->rank = rank;
  s->zsplit.assign(zsplit, zsplit + nranks + 1);
  s->split = KxSplit{nxh / nranks, nxh % nranks};
  s->nx = nx; s->ny = ny; s->nz = nz; s->nzl = nzl; s->nxh = nxh; s->npairs = npairs;
  s->kx0 = s->split.first(rank);
  s->nkx = s->split.count(rank);
  s->n = (long long)nx * ny * nz;
  s->n2d = (long long)nzl * ny * nxh;
  s->ncol = (long long)nz * ny * s->nkx;
  std::vector<int> sa(npairs), sb(npairs);
  std::vector<double> sc(npairs, 1.0);
  auto slot = [&](int v) {
    for (size_t i = 0; i < s->vars.size(); ++i) if (s->vars[i] == v) return (int)i;
    s->vars.push_back(v);
    return (int)s->vars.size() - 1;
  };
  for (int p = 0; p < npairs; ++p) {
    sa[p] = slot(pairA[p]);
    sb[p] = slot(pairB[p]);
    if (var_scaling) sc[p] = var_scaling[p];
  }
  s->nvars = (int)s->vars.size();
  // output column x holds frequency kx = x - nx/2 (mod nx); it is written from the half spectrum at kx, or at its partner nx - kx
  for (int x = 0; x < nx; ++x) {
    const int kx = (x + nx - nx / 2) % nx, k = kx < nxh ? kx : nx - kx;
    if (k >= s->kx0 && k < s->kx0 + s->nkx) s->colx.push_back(x);
  }
#define SF_TRY(x) do { int rc_ = (x); if (rc_) { bflbm_sf_slab_destroy(s); return rc_; } } while (0)
  SF_TRY([&]() -> int { SF_CU(cudaSetDevice(s->device)); return 0; }());
  auto alloc = [&](void** p, size_t bytes) -> int { SF_CU(cudaMalloc(p, bytes)); return 0; };
  const size_t cz = sizeof(cufftDoubleComplex);
  SF_TRY(alloc((void**)&s->hydro, (size_t)BFLBM_NHYDRO * nx * ny * nzl * sizeof(double)));
  SF_TRY(alloc((void**)&s->out2d, (size_t)s->n2d * cz));
  SF_TRY(alloc((void**)&s->send, (size_t)s->n2d * cz));
  SF_TRY(alloc((void**)&s->recv, (size_t)s->ncol * cz));
  SF_TRY(alloc((void**)&s->spec, (size_t)s->nvars * s->ncol * cz));
  SF_TRY(alloc((void**)&s->acc_re, (size_t)npairs * s->ncol * sizeof(double)));
  SF_TRY(alloc((void**)&s->acc_im, (size_t)npairs * s->ncol * sizeof(double)));
  SF_TRY(alloc((void**)&s->scale, npairs * sizeof(double)));
  SF_TRY(alloc((void**)&s->slotA, npairs * sizeof(int)));
  SF_TRY(alloc((void**)&s->slotB, npairs * sizeof(int)));
  SF_TRY(alloc((void**)&s->d_colx, s->colx.size() * sizeof(int)));
  SF_TRY([&]() -> int {
    SF_CU(cudaMemcpy(s->scale, sc.data(), npairs * sizeof(double), cudaMemcpyHostToDevice));
    SF_CU(cudaMemcpy(s->slotA, sa.data(), npairs * sizeof(int), cudaMemcpyHostToDevice));
    SF_CU(cudaMemcpy(s->slotB, sb.data(), npairs * sizeof(int), cudaMemcpyHostToDevice));
    SF_CU(cudaMemcpy(s->d_colx, s->colx.data(), s->colx.size() * sizeof(int), cudaMemcpyHostToDevice));
    return 0;
  }());
  // plans without their own work areas: one area, the larger of the two, serves both (they run one after the other on the stream)
  size_t ws2d = 0, wsz = 0;
  {
    long long n2[2] = {ny, nx};
    long long nzz[1] = {nz};
    const long long cstride = (long long)ny * s->nkx;
    bool ok = cufftCreate(&s->plan2d) == CUFFT_SUCCESS;
    s->have2d = ok;
    ok = ok && cufftSetAutoAllocation(s->plan2d, 0) == CUFFT_SUCCESS &&
         cufftMakePlanMany64(s->plan2d, 2, n2, nullptr, 1, (long long)ny * nx, nullptr, 1, (long long)ny * nxh, CUFFT_D2Z, nzl, &ws2d) == CUFFT_SUCCESS;
    ok = ok && cufftCreate(&s->planz) == CUFFT_SUCCESS;
    s->havez = ok;
    ok = ok && cufftSetAutoAllocation(s->planz, 0) == CUFFT_SUCCESS &&
         cufftMakePlanMany64(s->planz, 1, nzz, nzz, cstride, 1, nzz, cstride, 1, CUFFT_Z2Z, cstride, &wsz) == CUFFT_SUCCESS;
    if (!ok) { bflbm_sf_slab_destroy(s); return sf_fail(BFLBM_ERR_CUDA, "cuFFT plan creation failed"); }
  }
  const size_t ws = std::max(ws2d, wsz);
  if (ws) SF_TRY(alloc(&s->work, ws));
  if (cufftSetWorkArea(s->plan2d, s->work) != CUFFT_SUCCESS || cufftSetWorkArea(s->planz, s->work) != CUFFT_SUCCESS) {
    bflbm_sf_slab_destroy(s);
    return sf_fail(BFLBM_ERR_CUDA, "cufftSetWorkArea failed");
  }
  SF_TRY(bflbm_sf_slab_set_stream(s, nullptr));
  SF_TRY(bflbm_sf_slab_reset(s));
  SF_TRY([&]() -> int { SF_CU(cudaStreamSynchronize(s->stream)); return 0; }());
#undef SF_TRY
  *out = s;
  return 0;
}

int bflbm_sf_slab_set_stream(bflbm_sf_slab* s, void* cuda_stream) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  SF_CU(cudaSetDevice(s->device));
  SF_CU(cudaStreamSynchronize(s->stream));
  s->stream = (cudaStream_t)cuda_stream;
  if (cufftSetStream(s->plan2d, s->stream) != CUFFT_SUCCESS || cufftSetStream(s->planz, s->stream) != CUFFT_SUCCESS)
    return sf_fail(BFLBM_ERR_CUDA, "cufftSetStream failed");
  return 0;
}

int bflbm_sf_slab_rounds(const bflbm_sf_slab* s) { return s ? s->nvars : sf_fail(BFLBM_ERR_ARG, "null handle"); }

int bflbm_sf_slab_layout(const bflbm_sf_slab* s, int round, size_t* send_counts, size_t* send_displs, size_t* recv_counts,
                         size_t* recv_displs) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  if (round < 0 || round >= s->nvars) return sf_fail(BFLBM_ERR_ARG, "round outside [0, rounds)");
  // every round moves one variable, so the layout is the same for all of them
  const size_t rows = (size_t)s->nzl * s->ny;
  for (int r = 0; r < s->nranks; ++r) {
    const size_t zl = (size_t)(s->zsplit[r + 1] - s->zsplit[r]);
    if (send_counts) send_counts[r] = 2 * rows * s->split.count(r);
    if (send_displs) send_displs[r] = 2 * rows * s->split.first(r);
    if (recv_counts) recv_counts[r] = 2 * zl * s->ny * s->nkx;
    if (recv_displs) recv_displs[r] = 2 * (size_t)s->zsplit[r] * s->ny * s->nkx;
  }
  return 0;
}

void* bflbm_sf_slab_send_buffer(bflbm_sf_slab* s) { return s ? (void*)s->send : nullptr; }
void* bflbm_sf_slab_recv_buffer(bflbm_sf_slab* s) { return s ? (void*)s->recv : nullptr; }

int bflbm_sf_slab_begin(bflbm_sf_slab* s, int round) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  if (round < 0 || round >= s->nvars) return sf_fail(BFLBM_ERR_ARG, "round outside [0, rounds)");
  if (s->open_round >= 0 || round != s->next_round) return sf_fail(BFLBM_ERR_STATE, "rounds out of order");
  SF_CU(cudaSetDevice(s->device));
  if (round == 0) {
    // the observer runs on the lattice's stream: the previous accumulate's transforms must be done with the fields first
    SF_CU(cudaStreamSynchronize(s->stream));
    const int rc = bflbm_get_hydrovars_device(s->lat, s->hydro);
    if (rc) return sf_fail(rc, bflbm_last_error());
  }
  const long long nloc = (long long)s->nx * s->ny * s->nzl;
  if (cufftExecD2Z(s->plan2d, s->hydro + (long long)s->vars[round] * nloc, s->out2d) != CUFFT_SUCCESS)
    return sf_fail(BFLBM_ERR_CUDA, "cufftExecD2Z failed");
  const int T = 256;
  k_sf_slab_pack<<<(unsigned)((s->n2d + T - 1) / T), T, 0, s->stream>>>((long long)s->nzl * s->ny, s->nxh, s->split, s->out2d, s->send);
  SF_CU(cudaGetLastError());
  s->open_round = round;
  return 0;
}

int bflbm_sf_slab_end(bflbm_sf_slab* s, int round) {
  if (!s) return sf_fail(BFLBM_ERR_ARG, "null handle");
  if (round < 0 || round >= s->nvars) return sf_fail(BFLBM_ERR_ARG, "round outside [0, rounds)");
  if (s->open_round != round) return sf_fail(BFLBM_ERR_STATE, "end without a matching begin");
  SF_CU(cudaSetDevice(s->device));
  if (cufftExecZ2Z(s->planz, s->recv, s->spec + (long long)round * s->ncol, CUFFT_FORWARD) != CUFFT_SUCCESS)
    return sf_fail(BFLBM_ERR_CUDA, "cufftExecZ2Z failed");
  s->open_round = -1;
  s->next_round = (round + 1) % s->nvars;
  if (round == s->nvars - 1) {
    const int T = 256;
    k_sf_accumulate<<<(unsigned)((s->ncol + T - 1) / T), T, 0, s->stream>>>(s->ncol, s->npairs, s->slotA, s->slotB, s->scale, s->spec,
                                                                            1.0 / (double)s->n, s->acc_re, s->acc_im);
    SF_CU(cudaGetLastError());
    ++s->samples;
  }
  return 0;
}

long long bflbm_sf_slab_samples(const bflbm_sf_slab* s) { return s ? s->samples : -1; }

int bflbm_sf_slab_kx_range(const bflbm_sf_slab* s, int rank, int* kx0, int* nkx) {
  if (!s || rank < 0 || rank >= s->nranks) return sf_fail(BFLBM_ERR_ARG, "bad argument");
  if (kx0) *kx0 = s->split.first(rank);
  if (nkx) *nkx = s->split.count(rank);
  return 0;
}

int bflbm_sf_slab_get(bflbm_sf_slab* s, int zero_avg, double* real, double* imag) {
  if (!s || !real) return sf_fail(BFLBM_ERR_ARG, "null argument");
  if (s->samples == 0) return sf_fail(BFLBM_ERR_STATE, "no samples accumulated");
  SF_CU(cudaSetDevice(s->device));
  const int ncols = (int)s->colx.size();
  const size_t m = (size_t)s->nz * s->ny * ncols;  // one pair's values on this rank's columns
  // contiguous runs of colx: the host arrays take them with one memcpy per (z, y) row and run
  struct Run { int c, x, len; };
  std::vector<Run> runs;
  for (int c = 0; c < ncols; ++c) {
    if (!runs.empty() && s->colx[c] == runs.back().x + runs.back().len) ++runs.back().len;
    else runs.push_back({c, s->colx[c], 1});
  }
  double* d = nullptr;
  SF_CU(cudaMalloc(&d, 2 * m * sizeof(double)));
  std::vector<double> h(2 * m);
  int rc = 0;
  const dim3 block(128), grid((ncols + 127) / 128, s->ny, s->nz);
  for (int p = 0; p < s->npairs && !rc; ++p) {
    k_sf_slab_expand<<<grid, block, 0, s->stream>>>(s->nx, s->ny, s->nz, s->nxh, s->kx0, s->nkx, ncols, s->d_colx,
                                                    s->acc_re + (long long)p * s->ncol, s->acc_im + (long long)p * s->ncol,
                                                    1.0 / (double)s->samples, zero_avg, d, d + m);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), d, 2 * m * sizeof(double), cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) {
      rc = sf_fail(BFLBM_ERR_CUDA, std::string("bflbm_sf_slab_get: ") + cudaGetErrorString(e));
      break;
    }
    for (int part = 0; part < (imag ? 2 : 1); ++part) {
      double* dst = (part ? imag : real) + (long long)p * s->n;
      const double* src = h.data() + part * m;
      for (long long row = 0; row < (long long)s->nz * s->ny; ++row)
        for (const Run& r : runs)
          std::copy(src + row * ncols + r.c, src + row * ncols + r.c + r.len, dst + row * s->nx + r.x);
    }
  }
  cudaFree(d);
  return rc;
}

}  // extern "C"
