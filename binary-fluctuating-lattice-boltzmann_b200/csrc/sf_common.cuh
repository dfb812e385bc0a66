// Shared by the structure-factor accumulators (sf.cu: whole box on one device; sf_slab.cu: a box split over ranks):
// the error helper and the kernel that adds A_k conj(B_k) of every pair to the running sums.
#pragma once
#include <cuda_runtime.h>
#include <cufft.h>
#include <stdio.h>
#include <string>

#include "../../include/bflbm.h"

namespace {
thread_local std::string g_sf_err;
int sf_fail(int code, const std::string& msg) {
  g_sf_err = msg;
  fprintf(stderr, "bflbm_sf: %s\n", msg.c_str());
  return code;
}
#define SF_CU(call)                                                                              \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess) return sf_fail(BFLBM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// acc_re/im[p][i] += scale_p * A[i] conj(B[i]) / N   on the half spectrum (nz, ny, nxh), or a rank's columns of it
__global__ void k_sf_accumulate(long long nhalf, int npairs, const int* __restrict__ slotA, const int* __restrict__ slotB,
                                const double* __restrict__ scale, const cufftDoubleComplex* __restrict__ spec, double inv_n,
                                double* __restrict__ acc_re, double* __restrict__ acc_im) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nhalf) return;
  for (int p = 0; p < npairs; ++p) {
    const cufftDoubleComplex a = spec[(long long)slotA[p] * nhalf + i], b = spec[(long long)slotB[p] * nhalf + i];
    const double s = scale[p] * inv_n;
    acc_re[(long long)p * nhalf + i] += s * (a.x * b.x + a.y * b.y);
    acc_im[(long long)p * nhalf + i] += s * (a.y * b.x - a.x * b.y);
  }
}
}  // namespace
