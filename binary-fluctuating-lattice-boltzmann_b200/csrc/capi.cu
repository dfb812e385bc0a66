// C ABI of the B200-native fluctuating binary D3Q19 step (see include/bflbm.h for the contract and the
// reference interface each entry point replaces).  Host-side orchestration only; all arithmetic is in
// kernels.cuh / fused.cuh.  There is deliberately no CPU path: without a CUDA device every call fails.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <array>
#include <map>
#include <new>
#include <string>
#include <vector>

#include "../../include/bflbm.h"
#include "droplet_fit.hpp"
#include "fused.cuh"
#include "kernels.cuh"

using namespace bflbm;

namespace {
thread_local std::string g_err;
int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CU(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess) return fail(BFLBM_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)
#define CHECK_H(h)                                        \
  if (!(h)) return fail(BFLBM_ERR_ARG, "null lattice handle")
}  // namespace

struct bflbm_lattice {
  Geom G{};
  bflbm_params prm{};
  DevParams dp{};
  int device = 0;
  bool whole_box = true;
  bool initialized = false;
  int algo = 0;  // 0 fused one-pass, 1 two-pass
  bool algo_auto = true;  // nobody asked for an algorithm or a tiling: small whole boxes (L2 resident, launch / latency bound) use
                          // the thread-per-cell two-pass kernels, everything else the fused brick kernel
  int lz_request = 0;
  int cta_threads = 256;  // threads per CTA of the fused kernel (BFLBM_CTA_THREADS=128|256)
  bool rate1_fast_path = true;  // use the rate == 1 specialisation when tau_f = tau_g = 1/2 (BFLBM_RATE1=0 disables it)
  long long step = 0;
  long long launches = 0;
  size_t bytes = 0;

  cudaStream_t stream = nullptr;
  bool own_stream = false;
  // slab step with the halo exchange overlapped: the first and last brick row, the slab-face fold and the packing run
  // on `stream` (where the caller then queues its NCCL send/recv); the interior rows run on `aux` meanwhile
  cudaStream_t aux = nullptr;
  cudaEvent_t ev_prev = nullptr, ev_ends = nullptr, ev_interior = nullptr;
  bool overlap = true;          // BFLBM_OVERLAP=0: everything on `stream`, exchange after the whole step kernel
  bool interior_pending = false;

  double* X[2] = {nullptr, nullptr};
  int cur = 0;
  double2* R = nullptr;

  // fused algorithm
  BrickGrid B{};
  double2* E[2] = {nullptr, nullptr};  // extended boxes of the last two steps (ping-pong): E[ecur] is the newest
  int ecur = 0;
  bool e_valid = false;        // E[ecur] holds the densities of the current state (the step kernel may fold from it)
  bool r_stale = false;        // R is current only on brick-face planes; k_fold<2>(E[ecur]) completes it on demand
  bool fold_in_staging = true; // BFLBM_FOLD_IN_STAGING=0: separate full fold pass every step (first design)

  // halo messages : [side] ; layout see pack_halo().  recv[] = parity-0 slots of the mailbox (caller-driven exchange)
  double* send[2] = {nullptr, nullptr};
  double* recv[2] = {nullptr, nullptr};
  size_t halo_doubles = 0;
  double* mailbox = nullptr;                  // see "halo messages" below
  double* peer_base[2] = {nullptr, nullptr};  // the neighbours' mailboxes as seen from this GPU
  bool peer_mode = false;
  unsigned long long halo_seq = 0;
  std::vector<std::string> ipc_keys;  // CUDA-IPC mappings this lattice holds a reference to

  // staging for host transfers and diagnostics
  double* stage = nullptr;
  size_t stage_doubles = 0;
  double* diag_partial = nullptr;
  unsigned long long* diag_count = nullptr;
  size_t diag_blocks = 0;

  // asynchronous host transfers (bflbm_stage_populations / bflbm_get_hydrovars*_async): a copy stream next to the lattice's
  // stream, a checkpoint-sized staging area (`pre`) and an output buffer (`post`) on the device, all created on first use
  cudaStream_t cpy = nullptr;
  cudaEvent_t ev_staged = nullptr, ev_pre_free = nullptr, ev_observed = nullptr, ev_downloaded = nullptr;
  double* pre = nullptr;
  size_t pre_doubles = 0;
  int pre_state = 0;           // 0 nothing staged, 1 plain arrays, 2 ghosted arrays
  bool pre_consumed_once = false;
  double* post = nullptr;
  size_t post_doubles = 0;
  bool download_pending = false;

  dim3 block, grid_xy;  // thread-per-cell kernels: grid = (grid_xy.x, grid_xy.y, planes)

  // CUDA graphs of K consecutive whole-box steps (launch-bound small lattices: Parameters:1-37 runs 32^3 .. 8x256x64 boxes
  // for 1e5..1e6 steps).  Key = (K, cur, ecur); the step counter of the noise key lives in device memory (d_step) so that a
  // captured chunk can be replayed; d_step_host mirrors the value it will have once everything queued has run.
  bool use_graphs = true;  // BFLBM_GRAPH=0 disables
  std::map<long long, cudaGraphExec_t> graphs;
  std::map<long long, long long> graph_nodes;  // kernel nodes per graph (launch bookkeeping)
  long long* d_step = nullptr;
  long long d_step_host = -1;
  bool in_graph_capture = false;
  int graph_step_off = 0, graph_bump = 0;
  bool wrapped_in_fold = false;
  bool ghosts_stale = false;  // two-pass steps leave the ghost planes of X and R behind

  // what the last step launched (bflbm_debug_last_step), written on the host where the step kernel is launched; a graph
  // keeps the record of its capture, which run_graph_chunk restores on every replay
  std::array<int, BFLBM_LAST_STEP_FIELDS> last_step{};
  bool last_step_set = false;
  std::map<long long, std::array<int, BFLBM_LAST_STEP_FIELDS>> graph_last_step;

  // USE_REF_STATE noise (LBM_binary.H:12, 92-107; bflbm_set_reference_state): equilibrium profiles [rho_eq | phi_eq | rhot_eq] of the
  // whole box, the centre of mass of rho_eq, and the integer shift (com - com_ref) the device recomputes after every step
  double* eq = nullptr;
  int* d_shift = nullptr;
  double com_ref[3] = {0., 0., 0.};
  bool ref_relative = true;  // false after an analytic init: those pass the ABSOLUTE centre of mass (LBM_binary.H:623-625)
  // brick-kernel path: per-plane sums {rho, rho x, rho y, rho z} of all nz_global planes (k_com_chunks + k_com_fold_chunks; zeros
  // outside a slab), and the per-chunk partial sums of this slab's planes behind them (com_part).
  // A slab's entries of the other slabs arrive through the caller's all-reduce; com_pending until bflbm_com_update.
  double* com = nullptr;
  double* com_part = nullptr;
  bool com_pending = false;

  // optional per-kernel timing: events ev[0..4] bracket {step kernel, fold, pack, unpack}
  bool profiling = false;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  // deferred mode (bflbm_set_profiling(h, 2)): one set of five events per step from a pool, read back only when the pool is
  // full or the totals are asked for -- no host synchronisation inside a timed region
  static constexpr int PROF_POOL_STEPS = 128;
  std::vector<cudaEvent_t> evpool;
  bool prof_deferred = false;
  int prof_slot = 0;
  double prof_ms[4] = {0., 0., 0., 0.};
  long long prof_steps = 0;
};

void release_ipc(bflbm_lattice* h);  // defined next to the peer API

namespace {

int ceil_div(int a, int b) { return (a + b - 1) / b; }

// the twelve variants of the step kernel for one CTA size (eight + four reference-state ones); F = kernel functor applied to each
template <int NT, class Fn>
cudaError_t for_each_fused(Fn fn) {
  cudaError_t e = cudaSuccess;
#define BFLBM_EACH(N, R1, FU, REF) if (e == cudaSuccess) e = fn((const void*)k_step_fused<N, R1, FU, NT, REF>, R1, N)
  BFLBM_EACH(false, false, false, false); BFLBM_EACH(false, false, true, false);
  BFLBM_EACH(false, true, false, false);  BFLBM_EACH(false, true, true, false);
  BFLBM_EACH(true, false, false, false);  BFLBM_EACH(true, false, true, false);
  BFLBM_EACH(true, true, false, false);   BFLBM_EACH(true, true, true, false);
  BFLBM_EACH(true, false, false, true);   BFLBM_EACH(true, false, true, true);
  BFLBM_EACH(true, true, false, true);    BFLBM_EACH(true, true, true, true);
#undef BFLBM_EACH
  return e;
}
// Dynamic shared memory of the fused kernels.  The attribute is per FUNCTION and process-wide, not per lattice, so it is
// set once to the largest need over every brick shape make_brick_grid can produce (tx = 8, 16, 32): lattices of different
// shape or tau can then coexist.
template <int NT>
size_t fused_smem_max(bool rate1, bool noise) {
  size_t m = 0;
  for (int tx = 8; tx <= 32; tx <<= 1) {
    BrickGrid B{};
    B.tx = tx; B.ty = NT / tx; B.ex = B.tx + 2; B.ey = B.ty + 2; B.pl = B.ex * B.ey;
    m = std::max(m, fused_smem_bytes(B, rate1, noise));
  }
  return m;
}
cudaError_t set_fused_smem() {
  static bool done[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess || (dev < 64 && done[dev])) return e;
  e = for_each_fused<128>([&](const void* k, bool rate1, bool noise) {
    return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fused_smem_max<128>(rate1, noise));
  });
  if (e == cudaSuccess)
    e = for_each_fused<256>([&](const void* k, bool rate1, bool noise) {
      return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fused_smem_max<256>(rate1, noise));
    });
  // BFLBM_CARVEOUT=<percent of the SM's shared memory>: experiment knob (the driver otherwise sizes the carve-out to the
  // resident CTAs' need; what is left of the 256 KB is L1)
  if (const char* cv = getenv("BFLBM_CARVEOUT")) {
    const int pct = atoi(cv);
    auto setc = [&](const void* k, bool, bool) { return cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, pct); };
    if (e == cudaSuccess) e = for_each_fused<128>(setc);
    if (e == cudaSuccess) e = for_each_fused<256>(setc);
  }
  if (e == cudaSuccess && dev < 64) done[dev] = true;
  return e;
}

inline void mark(bflbm_lattice* h, int i) {
  if (h->profiling) cudaEventRecord(h->prof_deferred ? h->evpool[(size_t)h->prof_slot * 5 + i] : h->ev[i], h->stream);
}
inline void profile_add(bflbm_lattice* h, const cudaEvent_t* ev) {
  for (int i = 0; i < 4; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev[i], ev[i + 1]) == cudaSuccess) h->prof_ms[i] += ms;
  }
  ++h->prof_steps;
}
// deferred mode: read back the steps recorded so far (synchronises on the last of them)
inline void profile_flush(bflbm_lattice* h) {
  if (!h->prof_deferred || h->prof_slot == 0) return;
  cudaEventSynchronize(h->evpool[(size_t)(h->prof_slot - 1) * 5 + 4]);
  for (int s = 0; s < h->prof_slot; ++s) profile_add(h, &h->evpool[(size_t)s * 5]);
  h->prof_slot = 0;
}
// call after mark(4): folds the four intervals of one step into the totals (mode 1 synchronises the stream every step,
// mode 2 only when its event pool is full)
inline void profile_collect(bflbm_lattice* h) {
  if (!h->profiling) return;
  if (h->prof_deferred) {
    if (++h->prof_slot == bflbm_lattice::PROF_POOL_STEPS) profile_flush(h);
    return;
  }
  cudaEventSynchronize(h->ev[4]);
  profile_add(h, h->ev);
}

int set_device(const bflbm_lattice* h) {
  CU(cudaSetDevice(h->device));
  return 0;
}

int validate_params(const bflbm_params* p) {
  if (!p) return fail(BFLBM_ERR_ARG, "null params");
  if (!(p->tau_f > 0.) || !(p->tau_g > 0.)) return fail(BFLBM_ERR_ARG, "tau_f and tau_g must be > 0");
  if (p->alpha1 != 0.) return fail(BFLBM_ERR_ARG, "alpha1 must be 0: it does not enter the reference dynamics (LBM_binary.H:256-257)");
  if (p->kBT < 0.) return fail(BFLBM_ERR_ARG, "kBT must be >= 0");
  if (!(p->kappa > 0.)) return fail(BFLBM_ERR_ARG, "kappa must be > 0");
  return 0;
}

void derive(bflbm_lattice* h) {
  const bflbm_params& p = h->prm;
  DevParams& d = h->dp;
  d.rate_f = 1. / (p.tau_f * (1. + 0.5 / p.tau_f));
  d.rate_g = 1. / (p.tau_g * (1. + 0.5 / p.tau_g));
  d.fric_f = 0.5 / (p.tau_f + 0.5);
  d.fric_g = 0.5 / (p.tau_g + 0.5);
  d.force_pf = 1. / (1. + 1. / (2. * p.tau_f));
  d.acc_coef = -(1. / 3.) * p.alpha0;
  const double lam = 1. / (p.tau_f + 0.5);
  const double A = 2. * (lam - 0.5 * lam * lam);
  d.amp_j = A * p.kBT;
  d.amp_s = A * p.kBT / (1. / 3.);
  d.sqrt_amp_j = sqrt(d.amp_j);
  d.sqrt_amp_s = sqrt(d.amp_s);
  d.keys = philox_key_schedule(p.seed);
}

template <class T>
int dev_alloc(bflbm_lattice* h, T** p, size_t count) {
  CU(cudaMalloc((void**)p, count * sizeof(T)));
  h->bytes += count * sizeof(T);
  return 0;
}

int ensure_stage(bflbm_lattice* h, size_t doubles) {
  if (h->stage_doubles >= doubles) return 0;
  if (h->stage) {
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaFree(h->stage));
    h->bytes -= h->stage_doubles * sizeof(double);
    h->stage = nullptr;
    h->stage_doubles = 0;
  }
  CU(cudaMalloc((void**)&h->stage, doubles * sizeof(double)));
  h->stage_doubles = doubles;
  h->bytes += doubles * sizeof(double);
  return 0;
}

// planes per chunk so that ncomp*planes*plane doubles stay below 1 GiB
int chunk_planes(const bflbm_lattice* h, int ncomp, int extra_planes) {
  const size_t budget = (size_t)128 << 20;  // doubles (1 GiB stage)
  long long per_plane = (long long)ncomp * h->G.plane;
  long long n = (long long)(budget / (size_t)per_plane) - extra_planes;
  if (n < 1) n = 1;
  if (n > h->G.nzl) n = h->G.nzl;
  return (int)n;
}

dim3 cell_grid(const bflbm_lattice* h, int planes) { return dim3(h->grid_xy.x, h->grid_xy.y, planes); }
RefState rs_of(const bflbm_lattice* h) { return RefState{h->eq, h->d_shift}; }
int ensure_full_R(bflbm_lattice* h);
// the shift from the per-plane sums in h->com (all planes present: a whole box, or a slab after the caller's all-reduce)
int ref_com_shift(bflbm_lattice* h) {
  const double cx = h->ref_relative ? h->com_ref[0] : 0., cy = h->ref_relative ? h->com_ref[1] : 0., cz = h->ref_relative ? h->com_ref[2] : 0.;
  k_com_shift_planes<<<1, 1, 0, h->stream>>>(h->com, h->G.nz_global, cx, cy, cz, h->d_shift);
  ++h->launches;
  CU(cudaGetLastError());
  h->com_pending = false;
  return 0;
}
// update_com + shift for the reference-state noise.  Two-pass kernels (whole box): k_diag over R, which they keep complete.
// Brick kernels: R completed by the fold, then per-plane sums; a whole box takes the shift at once, a slab after the exchange.
int update_ref_shift(bflbm_lattice* h) {
  if (!h->eq) return 0;
  if (h->algo == 1) {
    k_diag<<<cell_grid(h, h->G.nzl), h->block, 0, h->stream>>>(h->G, h->R, h->diag_partial, h->diag_count);
    const double cx = h->ref_relative ? h->com_ref[0] : 0., cy = h->ref_relative ? h->com_ref[1] : 0., cz = h->ref_relative ? h->com_ref[2] : 0.;
    k_com_shift<<<1, 256, 0, h->stream>>>(h->diag_partial, (long long)h->diag_blocks, cx, cy, cz, h->d_shift);
    h->launches += 2;
    CU(cudaGetLastError());
    return 0;
  }
  int rc = ensure_full_R(h);
  if (rc) return rc;
  const int nchunk = com_chunks(h->G);
  k_com_chunks<<<dim3(nchunk, h->G.nzl), COM_THREADS, 0, h->stream>>>(h->G, h->R, h->com_part);
  k_com_fold_chunks<<<(h->G.nz_global + 127) / 128, 128, 0, h->stream>>>(h->G, h->com_part, nchunk, h->com);
  h->launches += 2;
  CU(cudaGetLastError());
  if (!h->whole_box) {
    h->com_pending = true;
    return 0;
  }
  return ref_com_shift(h);
}

// ---- ghost planes of a whole-box lattice (periodic in z inside one GPU) --------------------------------
int wrap_population_ghosts(bflbm_lattice* h, double* X) {
  const Geom& G = h->G;
  CopyList L;
  L.n = 0;
  for (int s = 0; s < 2; ++s)
    for (int i = 0; i < Q; ++i) {
      const long long base = (long long)(s * Q + i) * G.comp;
      if (cz(i) == 1) {  // pulled from plane below: ghost plane 0 <- plane nzl
        L.src[L.n] = base + (long long)G.nzl * G.plane;
        L.dst[L.n] = base;
        ++L.n;
      } else if (cz(i) == -1) {  // ghost plane nzl+1 <- plane 1
        L.src[L.n] = base + G.plane;
        L.dst[L.n] = base + (long long)(G.nzl + 1) * G.plane;
        ++L.n;
      }
    }
  const int T = 256;
  dim3 grid((unsigned)((G.plane + T - 1) / T), L.n);
  k_copy_planes<<<grid, T, 0, h->stream>>>(L, X, X, G.plane);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}
int wrap_density_ghosts(bflbm_lattice* h) {
  const Geom& G = h->G;
  CopyList L;
  L.n = 2;
  L.src[0] = 2 * (long long)G.nzl * G.plane; L.dst[0] = 0;
  L.src[1] = 2 * G.plane;                    L.dst[1] = 2 * (long long)(G.nzl + 1) * G.plane;
  const int T = 256;
  dim3 grid((unsigned)((2 * G.plane + T - 1) / T), L.n);
  k_copy_planes<<<grid, T, 0, h->stream>>>(L, (const double*)h->R, (double*)h->R, 2 * G.plane);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}
// ---- halo messages ------------------------------------------------------------------------------------
// Layout and protocol: fused.cuh (HaloPack / HaloUnpack).  SURVEY.md 8(e) option (ii), folded into a single message of
// 112 B per face cell per neighbour.  One pack launch and one unpack launch per step.
//
// Mailbox (one cudaMalloc per slab lattice, so that ONE CUDA-IPC handle exports it):
//   double recv[2 parities][2 sides][14 * plane]   incoming messages, double buffered by sequence parity
//   u64    flag[2 sides]                           sequence number of the newest complete message per side
//   u32    done, i32 err                           CTA counter of my pack kernel; set by a timed-out wait
// Peer mode (bflbm_peer_connect*): my message for the neighbour on `side` is written by the pack kernel straight into
// THAT lattice's recv[seq & 1][1 - side], then its flag[1 - side] <- seq.  Why two parities are enough: I overwrite a
// slot at exchange q + 2, after my wait for q + 1 has seen the neighbour's pack q + 1, which follows its unpack q on
// its stream.
size_t mailbox_recv_doubles(const bflbm_lattice* h) { return (size_t)4 * h->halo_doubles; }
size_t mailbox_bytes(const bflbm_lattice* h) { return mailbox_recv_doubles(h) * sizeof(double) + 64; }
double* mailbox_recv(double* base, const bflbm_lattice* h, int parity, int side) { return base + (size_t)(parity * 2 + side) * h->halo_doubles; }
unsigned long long* mailbox_flag(double* base, const bflbm_lattice* h, int side) {
  return reinterpret_cast<unsigned long long*>(base + mailbox_recv_doubles(h)) + side;
}
unsigned int* mailbox_done(double* base, const bflbm_lattice* h) { return reinterpret_cast<unsigned int*>(mailbox_flag(base, h, 0) + 2); }
int* mailbox_err(double* base, const bflbm_lattice* h) { return reinterpret_cast<int*>(mailbox_done(base, h) + 1); }

int pack_halo(bflbm_lattice* h) {
  const Geom& G = h->G;
  HaloPack P{};
  ++h->halo_seq;
  const int parity = (int)(h->halo_seq & 1);
  for (int side = 0; side < 2; ++side) {
    const int want = side == 0 ? -1 : 1;  // side 0: c_z = -1 of plane 0;  side 1: c_z = +1 of plane nzl-1
    const long long bplane = side == 0 ? 1 : G.nzl;  // storage index of my boundary plane
    int n = 0;
    for (int s = 0; s < 2; ++s)
      for (int i = 0; i < Q; ++i)
        if (cz(i) == want) P.pop_src[side][n++] = (long long)(s * Q + i) * G.comp + bplane * G.plane;
    // density partial planes: Pz = R[boundary], Ez = R[outside ghost] (local sums written by the fold)
    P.r_bnd[side] = 2 * bplane * G.plane;
    P.r_out[side] = 2 * (side == 0 ? 0 : (long long)(G.nzl + 1)) * G.plane;
    if (h->peer_mode) {
      P.dst[side] = mailbox_recv(h->peer_base[side], h, parity, 1 - side);
      P.flag[side] = mailbox_flag(h->peer_base[side], h, 1 - side);
    } else {
      P.dst[side] = h->send[side];
      P.flag[side] = nullptr;
    }
  }
  P.seq = h->halo_seq;
  P.done = mailbox_done(h->mailbox, h);
  const dim3 grid((unsigned)((G.plane + 256 * HALO_PER_THREAD - 1) / (256 * HALO_PER_THREAD)), 14, 2);
  k_pack_halo<<<grid, 256, 0, h->stream>>>(P, h->X[h->cur], (const double*)h->R, G.plane);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}
// recv[side] holds the message the neighbour on `side` packed for me (its side 1-side message); peer mode reads the mailbox
int unpack_halo(bflbm_lattice* h, double* const recv[2]) {
  const Geom& G = h->G;
  HaloUnpack U{};
  const int parity = (int)(h->halo_seq & 1);
  for (int side = 0; side < 2; ++side) {
    // lower neighbour sent its c_z = +1 populations (its side-1 message): they go to my ghost plane 0
    const int want = side == 0 ? 1 : -1;
    const long long gplane = side == 0 ? 0 : G.nzl + 1, bplane = side == 0 ? 1 : G.nzl;
    int n = 0;
    for (int s = 0; s < 2; ++s)
      for (int i = 0; i < Q; ++i)
        if (cz(i) == want) U.pop_dst[side][n++] = (long long)(s * Q + i) * G.comp + gplane * G.plane;
    U.r_bnd[side] = bplane * G.plane;
    U.r_ghost[side] = gplane * G.plane;
    if (h->peer_mode) {
      U.src[side] = mailbox_recv(h->mailbox, h, parity, side);
      U.flag[side] = mailbox_flag(h->mailbox, h, side);
    } else {
      U.src[side] = recv[side];
      U.flag[side] = nullptr;
    }
  }
  U.seq = h->halo_seq;
  U.err = mailbox_err(h->mailbox, h);
  const dim3 grid((unsigned)((G.plane + 256 * HALO_PER_THREAD - 1) / (256 * HALO_PER_THREAD)), 11, 2);
  k_unpack_halo<<<grid, 256, 0, h->stream>>>(U, h->X[h->cur], h->R, G.plane);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}

// mode 0: all planes; 1: brick-face planes + slab-face outputs; 2: the complement of 1
// 3: the four slab-face planes (first / last brick row only); 4 = 1 without 3
int fold_local(bflbm_lattice* h, int mode, cudaStream_t st = nullptr) {
  const Geom& G = h->G;
  if (!st) st = h->stream;
  const dim3 grid(h->B.bx, h->B.by, mode == 3 ? std::min(2, h->B.bz) : h->B.bz), block(h->B.tx, h->B.ty);
  if (mode == 0)      k_fold<0><<<grid, block, 0, st>>>(G, h->B, h->E[h->ecur], h->R);
  else if (mode == 1) k_fold<1><<<grid, block, 0, st>>>(G, h->B, h->E[h->ecur], h->R);
  else if (mode == 2) k_fold<2><<<grid, block, 0, st>>>(G, h->B, h->E[h->ecur], h->R);
  else if (mode == 3) k_fold<3><<<grid, block, 0, st>>>(G, h->B, h->E[h->ecur], h->R);
  else                k_fold<4><<<grid, block, 0, st>>>(G, h->B, h->E[h->ecur], h->R);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}
// whole box: brick-face fold + periodic self-exchange (densities and population ghost planes) in one launch;
// bump > 0 (last step of a graph chunk): advance the device-side step counter
int fold_wrap_whole_box(bflbm_lattice* h, int bump) {
  const dim3 grid(h->B.bx, h->B.by, h->B.bz + 1), block(h->B.tx, h->B.ty);
  k_fold<5><<<grid, block, 0, h->stream>>>(h->G, h->B, h->E[h->ecur], h->R, h->X[h->cur], bump > 0 ? h->d_step : nullptr, bump);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}
// R complete on every plane (observers, diagnostics, kernels that stage every plane from R)
int ensure_full_R(bflbm_lattice* h) {
  if (!h->r_stale) return 0;
  int rc = fold_local(h, 2);
  if (rc) return rc;
  h->r_stale = false;
  return 0;
}

// the fields of bflbm_debug_last_step, in its order (include/bflbm.h)
void record_step(bflbm_lattice* h, int algo, int threads, int tile_x, int tile_y, int lz, int nbx, int nby, int nbz, bool full,
                 bool rate1, bool noise, bool staged_from_e, int schedule) {
  h->last_step = {algo, threads, tile_x, tile_y, lz, nbx, nby, nbz, full, rate1, noise, staged_from_e, schedule, h->in_graph_capture};
  h->last_step_set = true;
}

// rows: 0 = every brick row, 1 = the first and the last row (two z-blocks), 2 = rows 1 .. bz-2
template <bool NOISE, bool R1, bool FU, bool REF>
int launch_fused_v(bflbm_lattice* h, int rows, cudaStream_t st) {
  const BrickGrid& B = h->B;
  const dim3 grid(B.bx, B.by, rows == 0 ? B.bz : (rows == 1 ? 2 : B.bz - 2)), block(B.tx, B.ty);
  const int bz0 = rows == 2 ? 1 : 0, two_ends = rows == 1;
  const double2* Ein = (h->e_valid && h->fold_in_staging) ? h->E[h->ecur] : nullptr;
  record_step(h, 0, B.tx * B.ty, B.tx, B.ty, B.lz, B.bx, B.by, B.bz, FU, R1, NOISE, Ein != nullptr, rows != 0 ? 2 : (h->whole_box ? 0 : 1));
  double2* Eout = h->E[1 - h->ecur];
  const PopBases XB = make_pop_bases(h->G, h->X[h->cur], h->X[1 - h->cur]);
  // inside a graph capture the step is (device counter) + (offset in the chunk); otherwise it is passed by value
  const long long step = h->in_graph_capture ? (long long)h->graph_step_off : h->step;
  const long long* sdev = h->in_graph_capture ? h->d_step : nullptr;
  const RefState RS = rs_of(h);
  if (B.tx * B.ty == 128)
    k_step_fused<NOISE, R1, FU, 128, REF><<<grid, block, fused_smem_bytes(B, R1, NOISE), st>>>(h->G, B, h->dp, step, sdev, XB, h->R, Ein, Eout, bz0, two_ends, RS);
  else
    k_step_fused<NOISE, R1, FU, 256, REF><<<grid, block, fused_smem_bytes(B, R1, NOISE), st>>>(h->G, B, h->dp, step, sdev, XB, h->R, Ein, Eout, bz0, two_ends, RS);
  ++h->launches;
  CU(cudaGetLastError());
  return 0;
}
template <bool NOISE, bool REF>
int launch_fused_r(bflbm_lattice* h, int rows, cudaStream_t st) {
  const bool rate1 = h->rate1_fast_path && h->dp.rate_f == 1. && h->dp.rate_g == 1.;
  const bool full = h->G.nx % h->B.tx == 0 && h->G.ny % h->B.ty == 0;
  if (rate1) return full ? launch_fused_v<NOISE, true, true, REF>(h, rows, st) : launch_fused_v<NOISE, true, false, REF>(h, rows, st);
  return full ? launch_fused_v<NOISE, false, true, REF>(h, rows, st) : launch_fused_v<NOISE, false, false, REF>(h, rows, st);
}
// the reference state changes the noise amplitudes only: without noise the plain kernels run
template <bool NOISE>
int launch_fused(bflbm_lattice* h, int rows, cudaStream_t st) {
  if constexpr (NOISE) {
    if (h->eq) return launch_fused_r<true, true>(h, rows, st);
  }
  return launch_fused_r<NOISE, false>(h, rows, st);
}

// LBM_timestep passes com - com_ref (LBM_binary.H:586-588)
int ref_shift_after_step(bflbm_lattice* h) {
  h->ref_relative = true;
  return update_ref_shift(h);
}

// collide+stream of the slab and local density partials; leaves the outgoing messages packed
int step_local(bflbm_lattice* h, bool pack = true) {
  const bool noise = h->prm.kBT > 0.;
  mark(h, 0);
  int rc0 = 0;
  // every kernel but the default one stages all planes from R; the default one only when E is not usable
  if ((h->algo != 0 || !h->e_valid || !h->fold_in_staging) && (rc0 = ensure_full_R(h))) return rc0;
  if (h->algo == 1) {
    // whole box only: z wraps by index arithmetic (Geom::zwrap), so a step is exactly two launches and no ghost plane is
    // read or written; they are refreshed when the lattice goes back to the fused kernel (bflbm_set_algorithm)
    h->e_valid = false;
    const long long step = h->in_graph_capture ? (long long)h->graph_step_off : h->step;
    const long long* sdev = h->in_graph_capture ? h->d_step : nullptr;
    const bool rate1 = h->rate1_fast_path && h->dp.rate_f == 1. && h->dp.rate_g == 1.;
    const dim3 grid = cell_grid(h, h->G.nzl);
    record_step(h, 1, h->block.x * h->block.y, h->block.x, h->block.y, 1, grid.x, grid.y, grid.z, false, rate1, noise, false, 0);
#define BFLBM_TP(N, R1) k_step_twopass<N, R1><<<grid, h->block, 0, h->stream>>>(h->G, h->dp, step, sdev, h->X[h->cur], h->X[1 - h->cur], h->R, rs_of(h))
    if (noise) { if (rate1) BFLBM_TP(true, true); else BFLBM_TP(true, false); }
    else       { if (rate1) BFLBM_TP(false, true); else BFLBM_TP(false, false); }
#undef BFLBM_TP
    ++h->launches;
    CU(cudaGetLastError());
    h->cur ^= 1;
    h->ghosts_stale = true;
    mark(h, 1);
    k_density<<<cell_grid(h, h->G.nzl), h->block, 0, h->stream>>>(h->G, h->X[h->cur], h->R, h->graph_bump > 0 ? h->d_step : nullptr, h->graph_bump);
    ++h->launches;
    CU(cudaGetLastError());
    if ((rc0 = ref_shift_after_step(h))) return rc0;
    mark(h, 2);
    mark(h, 3);
    return 0;
  }
  if (h->ghosts_stale) {  // two-pass steps were taken: the brick kernel reads ghost planes again
    int rcg;
    if ((rcg = wrap_population_ghosts(h, h->X[h->cur])) || (rcg = wrap_density_ghosts(h))) return rcg;
    h->ghosts_stale = false;
  }
  // the default kernel folds the brick-interior planes itself while staging (next step): only the brick faces here
  const bool partial = h->algo == 0 && h->fold_in_staging && fold_in_staging_ok(h->G, h->B);
  int rc;
  // The overlapped schedule needs a last brick row of at least two planes: with a single plane, the slab-face fold on
  // `stream` would read the top shell of row bz-2 while `aux` is still writing it (and overwrite the R plane that row
  // stages for its top gradients).  Such slabs take the single-stream path below.
  const bool last_row_ok = h->G.nzl - (h->B.bz - 1) * h->B.lz >= 2;
  if (!h->whole_box && h->overlap && !h->profiling && partial && h->B.bz >= 3 && last_row_ok) {
    // overlapped slab step.  stream: [first+last brick row] -> [fold of the 4 slab-face planes] -> [pack] -> caller's
    // exchange -> (step_end) unpack.  aux: [interior rows] -> [fold of the other brick faces], concurrent with the exchange.
    CU(cudaEventRecord(h->ev_prev, h->stream));          // everything queued so far (previous step, uploads, observers)
    CU(cudaStreamWaitEvent(h->aux, h->ev_prev, 0));
    if ((rc = noise ? launch_fused<true>(h, 1, h->stream) : launch_fused<false>(h, 1, h->stream))) return rc;
    CU(cudaEventRecord(h->ev_ends, h->stream));
    if ((rc = noise ? launch_fused<true>(h, 2, h->aux) : launch_fused<false>(h, 2, h->aux))) return rc;
    h->cur ^= 1;
    h->ecur ^= 1;
    h->e_valid = true;
    h->r_stale = true;
    if ((rc = fold_local(h, 3))) return rc;
    if ((rc = pack_halo(h))) return rc;
    CU(cudaStreamWaitEvent(h->aux, h->ev_ends, 0));      // the brick faces next to the end rows need their extended boxes
    if ((rc = fold_local(h, 4, h->aux))) return rc;
    CU(cudaEventRecord(h->ev_interior, h->aux));
    h->interior_pending = true;
    return 0;
  }
  rc = noise ? launch_fused<true>(h, 0, h->stream) : launch_fused<false>(h, 0, h->stream);
  if (rc) return rc;
  h->cur ^= 1;
  h->ecur ^= 1;
  mark(h, 1);
  h->e_valid = partial;
  h->r_stale = partial;
  // whole box stepped by bflbm_step: the brick-face fold and the periodic self-exchange are one launch
  h->wrapped_in_fold = h->whole_box && !pack && partial;
  if ((rc = h->wrapped_in_fold ? fold_wrap_whole_box(h, h->graph_bump) : fold_local(h, partial ? 1 : 0))) return rc;
  mark(h, 2);
  if (pack) rc = pack_halo(h);
  // reference state on a whole box whose step is complete here (also inside a graph capture): the centre of mass for the next
  // step; it takes the third profiling interval, which such a step leaves empty
  if (!rc && h->wrapped_in_fold && h->eq) rc = ref_shift_after_step(h);
  mark(h, 3);
  return rc;
}

__global__ void k_set_step(long long* p, long long v) { *p = v; }

void drop_graphs(bflbm_lattice* h) {
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second);
  h->graphs.clear();
}
bool graph_ok(const bflbm_lattice* h) {
  if (!h->use_graphs || !h->whole_box || h->profiling) return false;
  return h->algo == 1 || (h->e_valid && h->fold_in_staging && fold_in_staging_ok(h->G, h->B));
}
// K (even) whole-box steps as one graph launch; the graph is captured from the very launches step_local makes
int run_graph_chunk(bflbm_lattice* h, int K) {
  const long long key = ((long long)K << 3) | (h->algo << 2) | (h->cur << 1) | h->ecur;
  auto it = h->graphs.find(key);
  if (it == h->graphs.end()) {
    const long long launches0 = h->launches;
    cudaGraph_t g = nullptr;
    CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    h->in_graph_capture = true;
    int rc = 0;
    for (int j = 0; j < K && !rc; ++j) {
      h->graph_step_off = j;
      h->graph_bump = j == K - 1 ? K : 0;
      rc = step_local(h, /*pack=*/false);
    }
    h->in_graph_capture = false;
    h->graph_bump = 0;
    h->graph_nodes[key] = h->launches - launches0;
    h->graph_last_step[key] = h->last_step;
    h->launches = launches0;
    const cudaError_t e = cudaStreamEndCapture(h->stream, &g);
    if (rc || e != cudaSuccess || !g) {
      if (g) cudaGraphDestroy(g);
      cudaGetLastError();
      h->use_graphs = false;  // e.g. the caller's stream is itself being captured: plain launches from now on
      return rc ? rc : fail(BFLBM_ERR_CUDA, "graph capture: %s", cudaGetErrorString(e));
    }
    cudaGraphExec_t ex = nullptr;
    const cudaError_t e2 = cudaGraphInstantiate(&ex, g, 0);
    cudaGraphDestroy(g);
    if (e2 != cudaSuccess) { h->use_graphs = false; return fail(BFLBM_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e2)); }
    it = h->graphs.emplace(key, ex).first;
  }
  if (h->d_step_host != h->step) {
    k_set_step<<<1, 1, 0, h->stream>>>(h->d_step, h->step);
    ++h->launches;
    h->d_step_host = h->step;
  }
  CU(cudaGraphLaunch(it->second, h->stream));
  h->launches += h->graph_nodes[key];
  h->last_step = h->graph_last_step[key];
  h->last_step_set = true;
  h->step += K;
  h->d_step_host += K;
  if (h->algo == 0) {
    h->e_valid = true;
    h->r_stale = true;
  } else {
    h->ghosts_stale = true;
  }
  return 0;
}

int create_common(const bflbm_params* p, int nx, int ny, int nz_global, int z0, int nzl, int device, bool whole, bflbm_lattice** out) {
  if (!out) return fail(BFLBM_ERR_ARG, "null out pointer");
  *out = nullptr;
  int rc = validate_params(p);
  if (rc) return rc;
  if (nx < 1 || ny < 1 || nz_global < 2 || nzl < 2 || z0 < 0 || z0 + nzl > nz_global)
    return fail(BFLBM_ERR_ARG, "bad lattice size nx=%d ny=%d nz=%d z0=%d nz_local=%d (need nx,ny >= 1, nz_local >= 2)", nx, ny, nz_global, z0, nzl);
  if ((double)(nzl + 2) * nx * ny * 8.0 >= 4294967296.0)
    return fail(BFLBM_ERR_ARG, "slab too large: (nz_local+2)*nx*ny*8 B must stay below 4 GiB per component (32-bit in-component offsets); "
                               "use more slabs");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(BFLBM_ERR_CUDA, "no CUDA device available: this library has no CPU path");
  if (device < 0 || device >= ndev) return fail(BFLBM_ERR_ARG, "device %d out of range (have %d)", device, ndev);
  bflbm_lattice* h = new (std::nothrow) bflbm_lattice;
  if (!h) return fail(BFLBM_ERR_ARG, "out of host memory");
  h->device = device;
  h->whole_box = whole;
  h->prm = *p;
  h->step = p->step0;
  derive(h);
  Geom& G = h->G;
  G.nx = nx; G.ny = ny; G.nzl = nzl; G.nz_global = nz_global; G.z0 = z0;
  G.plane = (long long)nx * ny;
  G.comp = (long long)(nzl + 2) * G.plane;
  G.zwrap = whole ? 1 : 0;
  int bx = 8;
  while (bx < nx && bx < 128) bx <<= 1;
  h->block = dim3(bx, 256 / bx);
  h->grid_xy = dim3(ceil_div(nx, bx), ceil_div(ny, 256 / bx));
#define TRY(x) if ((rc = (x))) { bflbm_destroy(h); return rc; }
  TRY(set_device(h));
  {
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete h; return fail(BFLBM_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    h->own_stream = true;
  }
  TRY(dev_alloc(h, &h->X[0], (size_t)(2 * Q) * G.comp));
  TRY(dev_alloc(h, &h->X[1], (size_t)(2 * Q) * G.comp));
  TRY(dev_alloc(h, &h->R, (size_t)G.comp));
  {
    const char* nt = getenv("BFLBM_CTA_THREADS");
    h->cta_threads = (nt && atoi(nt) == 128) ? 128 : 256;
  }
  h->B = make_brick_grid(G, 0, h->cta_threads, 32);
  // a slab wants at least 3 brick rows so that the halo exchange can overlap the interior rows (thin strong-scaling slabs)
  while (!whole && h->B.bz < 3 && h->B.lz >= 16) h->B = make_brick_grid(G, h->B.lz / 2, h->cta_threads, 32);
  TRY(dev_alloc(h, &h->E[0], brick_doubles2(h->B)));
  TRY(dev_alloc(h, &h->E[1], brick_doubles2(h->B)));
  if (!whole) {
    const char* ov = getenv("BFLBM_OVERLAP");
    h->overlap = !(ov && ov[0] == '0');
    cudaError_t e = cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_prev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_ends, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_interior, cudaEventDisableTiming);
    if (e != cudaSuccess) { bflbm_destroy(h); return fail(BFLBM_ERR_CUDA, "aux stream / events: %s", cudaGetErrorString(e)); }
  }
  {
    const char* fs = getenv("BFLBM_FOLD_IN_STAGING");
    h->fold_in_staging = !(fs && fs[0] == '0');
  }
  h->halo_doubles = (size_t)14 * G.plane;
  for (int s = 0; s < 2; ++s) TRY(dev_alloc(h, &h->send[s], h->halo_doubles));
  {
    char* mb = nullptr;
    TRY(dev_alloc(h, &mb, mailbox_bytes(h)));
    h->mailbox = reinterpret_cast<double*>(mb);
    if (cudaMemset(mb, 0, mailbox_bytes(h)) != cudaSuccess) { bflbm_destroy(h); return fail(BFLBM_ERR_CUDA, "cudaMemset(mailbox)"); }
    for (int s = 0; s < 2; ++s) h->recv[s] = mailbox_recv(h->mailbox, h, 0, s);
  }
  {
    // automatic kernel choice (until the caller asks for an algorithm or a brick height): whole boxes small enough to live in
    // the 126 MB L2 are latency bound, not bandwidth bound -- the thread-per-cell two-pass kernels (2 launches, no barriers,
    // no per-CTA prologue) beat the brick sweep there; measured cross-over in profiles/README.md
    long long small = 150000;
    if (const char* sc = getenv("BFLBM_SMALL_CELLS")) small = atoll(sc);
    if (whole && (long long)nx * ny * nzl <= small) h->algo = 1;
  }
  TRY(dev_alloc(h, &h->d_step, (size_t)1));
  {
    const char* gr = getenv("BFLBM_GRAPH");
    h->use_graphs = !(gr && gr[0] == '0');
  }
  h->diag_blocks = (size_t)h->grid_xy.x * h->grid_xy.y * nzl;
  TRY(dev_alloc(h, &h->diag_partial, h->diag_blocks * NDIAG));
  TRY(dev_alloc(h, &h->diag_count, (size_t)1));
  {
    const char* r1 = getenv("BFLBM_RATE1");
    h->rate1_fast_path = !(r1 && r1[0] == '0');
    cudaError_t e = set_fused_smem();
    if (e != cudaSuccess) { bflbm_destroy(h); return fail(BFLBM_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); }
  }
#undef TRY
  *out = h;
  return 0;
}

// after X planes 1..nzl are set (whole box): make ghosts, densities consistent
int finish_init(bflbm_lattice* h) {
  h->step = h->prm.step0;
  h->initialized = true;
  h->e_valid = false;  // R was (or is about to be) rebuilt from the populations; E is void
  h->r_stale = false;
  h->ghosts_stale = false;
  return 0;
}

int run_init(bflbm_lattice* h, const InitSpec& S) {
  int rc = set_device(h);
  if (rc) return rc;
  k_init<<<cell_grid(h, h->G.nzl + 2), h->block, 0, h->stream>>>(h->G, S, h->X[h->cur], h->R);
  ++h->launches;
  CU(cudaGetLastError());
  if ((rc = finish_init(h))) return rc;
  h->ref_relative = false;  // the analytic inits hand thermal_noise the absolute centre of mass (LBM_binary.H:623-625)
  return update_ref_shift(h);
}

// generic chunked observer -> host (or device) array of ncomp components
template <int MODE>
int observe(bflbm_lattice* h, int ncomp, double* out, bool out_is_device, bool cell_major, bool into_global = false) {
  CHECK_H(h);
  if (!out) return fail(BFLBM_ERR_ARG, "null output buffer");
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  const Geom& G = h->G;
  const bool noise = h->prm.kBT > 0.;
  const int cp = chunk_planes(h, ncomp, 0);
  if ((rc = ensure_stage(h, (size_t)ncomp * cp * G.plane))) return rc;
  for (int zlo = 0; zlo < G.nzl; zlo += cp) {
    const int zc = std::min(cp, G.nzl - zlo);
    if (noise) k_observe<MODE, true><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    else       k_observe<MODE, false><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    ++h->launches;
    CU(cudaGetLastError());
    const cudaMemcpyKind kind = out_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    // into_global: `out` is an array of the WHOLE box (component stride nz_global planes); this slab fills its planes
    const size_t z_off = into_global ? (size_t)G.z0 : 0, comp_planes = into_global ? (size_t)G.nz_global : (size_t)G.nzl;
    if (cell_major) {
      CU(cudaMemcpyAsync(out + ((size_t)zlo + z_off) * G.plane * ncomp, h->stage, (size_t)zc * G.plane * ncomp * sizeof(double), kind, h->stream));
    } else {
      CU(cudaMemcpy2DAsync(out + ((size_t)zlo + z_off) * G.plane, comp_planes * G.plane * sizeof(double), h->stage,
                           (size_t)zc * G.plane * sizeof(double), (size_t)zc * G.plane * sizeof(double), ncomp, kind, h->stream));
    }
    // the stage is reused by the next chunk: stream order (kernel after copy) protects it, no host sync per chunk
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// Restart upload.  mode 0: whole box, host arrays (19, nzl, ny, nx).  mode 1: slab, ghosted host arrays (19, nzl+2, ny, nx).
// mode 2: slab (or whole box), host arrays of the WHOLE box (19, nz_global, ny, nx): the lattice takes its own planes and,
// for a slab, the two periodic neighbour planes.  Source planes are uploaded in chunks of up to 1 GiB and scattered to
// their (pre-stream) positions by k_scatter_populations.
int upload_populations(bflbm_lattice* h, const double* f, const double* g, int mode) {
  const Geom& G = h->G;
  int rc;
  const bool wrap = h->whole_box && mode != 1;  // targets wrap periodically inside the lattice; otherwise ghost planes are sources
  const int zfirst = wrap ? 0 : -1, nsrc = wrap ? G.nzl : G.nzl + 2;   // source planes zfirst .. zfirst + nsrc - 1 (local numbering)
  const size_t host_planes = mode == 0 ? (size_t)G.nzl : (mode == 1 ? (size_t)G.nzl + 2 : (size_t)G.nz_global);
  const size_t budget = (size_t)128 << 20;  // doubles (1 GiB): a few large copies per component instead of one per plane
  int cp = (int)std::max<size_t>(1, std::min<size_t>((size_t)nsrc, budget / ((size_t)(2 * Q) * (size_t)G.plane)));
  if ((rc = ensure_stage(h, (size_t)(2 * Q) * cp * G.plane))) return rc;
  const double* src[2] = {f, g};
  const size_t spitch = host_planes * G.plane * sizeof(double);
  // host plane index of local source plane zs
  auto host_plane = [&](int zs) -> long long {
    if (mode == 0) return zs;
    if (mode == 1) return zs + 1;
    long long zg = (long long)G.z0 + zs;
    return ((zg % G.nz_global) + G.nz_global) % G.nz_global;
  };
  for (int z = 0; z < nsrc;) {
    int zc = std::min(cp, nsrc - z);
    if (mode == 2) {  // a chunk must be contiguous in the global array: cut at the periodic wrap
      const long long hp = host_plane(zfirst + z);
      zc = (int)std::min<long long>(zc, G.nz_global - hp);
      if (!wrap && zfirst + z < 0) zc = 1;  // the lower ghost plane is a chunk of its own (its successor may wrap back to plane 0)
    }
    const size_t dpitch = (size_t)zc * G.plane * sizeof(double);
    for (int sp = 0; sp < 2; ++sp)
      CU(cudaMemcpy2DAsync(h->stage + (size_t)sp * Q * zc * G.plane, dpitch, src[sp] + (size_t)host_plane(zfirst + z) * G.plane, spitch, dpitch, Q,
                           cudaMemcpyHostToDevice, h->stream));
    // stream order protects the stage: the next chunk's copies start after this kernel has read it (no host sync)
    k_scatter_populations<<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, zfirst + z, wrap ? 1 : 0, h->stage, h->X[h->cur]);
    ++h->launches;
    CU(cudaGetLastError());
    z += zc;
  }
  CU(cudaStreamSynchronize(h->stream));  // the caller's host buffers are free again
  return 0;
}

// fold/gold or fnoisevs/gnoisevs: one observer pass produces both species (38 components), split into two host arrays
template <int MODE>
int observe_pair(bflbm_lattice* h, double* a, double* b, bool into_global) {
  CHECK_H(h);
  if (!a || !b) return fail(BFLBM_ERR_ARG, "null output buffer");
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  const Geom& G = h->G;
  const bool noise = MODE == OBS_NOISE && h->prm.kBT > 0.;
  const int cp = chunk_planes(h, 2 * Q, 0);
  if ((rc = ensure_stage(h, (size_t)(2 * Q) * cp * G.plane))) return rc;
  const size_t z_off = into_global ? (size_t)G.z0 : 0, comp_planes = into_global ? (size_t)G.nz_global : (size_t)G.nzl;
  for (int zlo = 0; zlo < G.nzl; zlo += cp) {
    const int zc = std::min(cp, G.nzl - zlo);
    if (noise) k_observe<MODE, true><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    else       k_observe<MODE, false><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    ++h->launches;
    CU(cudaGetLastError());
    double* outs[2] = {a, b};
    for (int s = 0; s < 2; ++s)
      CU(cudaMemcpy2DAsync(outs[s] + ((size_t)zlo + z_off) * G.plane, comp_planes * G.plane * sizeof(double), h->stage + (size_t)s * Q * zc * G.plane,
                           (size_t)zc * G.plane * sizeof(double), (size_t)zc * G.plane * sizeof(double), Q, cudaMemcpyDeviceToHost, h->stream));
    // the stage is reused by the next chunk: stream order (kernel after copy) protects it
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// ---- asynchronous host transfers ------------------------------------------------------------------------------------------
int ensure_copy_stream(bflbm_lattice* h) {
  if (h->cpy) return 0;
  CU(cudaStreamCreateWithFlags(&h->cpy, cudaStreamNonBlocking));
  for (cudaEvent_t* e : {&h->ev_staged, &h->ev_pre_free, &h->ev_observed, &h->ev_downloaded}) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  return 0;
}
int ensure_buffer(bflbm_lattice* h, double** buf, size_t* have, size_t doubles) {
  if (*have >= doubles) return 0;
  if (*buf) {
    CU(cudaStreamSynchronize(h->cpy));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaFree(*buf));
    h->bytes -= *have * sizeof(double);
    *buf = nullptr;
    *have = 0;
  }
  const cudaError_t e = cudaMalloc((void**)buf, doubles * sizeof(double));
  if (e != cudaSuccess) {  // not sticky: clear it, so that the next launch check does not report it again; the lattice stays usable
    cudaGetLastError();
    *buf = nullptr;
    return fail(BFLBM_ERR_CUDA, "asynchronous transfers: no room for %.2f GB of staging on the device (%s); the blocking calls need none",
                (double)doubles * 8e-9, cudaGetErrorString(e));
  }
  *have = doubles;
  h->bytes += doubles * sizeof(double);
  return 0;
}

// observer over the whole local lattice into `post` (component-major = the host layout), then ONE device -> host copy on the
// copy stream; steps queued on the lattice's stream afterwards run next to the copy
template <int MODE>
int observe_async(bflbm_lattice* h, int ncomp, double* out) {
  CHECK_H(h);
  if (!out) return fail(BFLBM_ERR_ARG, "null output buffer");
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_copy_stream(h))) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  const Geom& G = h->G;
  const size_t n = (size_t)ncomp * G.nzl * G.plane;
  if ((rc = ensure_buffer(h, &h->post, &h->post_doubles, n))) return rc;
  if (h->download_pending) CU(cudaStreamWaitEvent(h->stream, h->ev_downloaded, 0));  // `post` is still being read
  if (h->prm.kBT > 0.) k_observe<MODE, true><<<cell_grid(h, G.nzl), h->block, 0, h->stream>>>(G, h->dp, h->step, 0, h->X[h->cur], h->R, h->post, rs_of(h));
  else                 k_observe<MODE, false><<<cell_grid(h, G.nzl), h->block, 0, h->stream>>>(G, h->dp, h->step, 0, h->X[h->cur], h->R, h->post, rs_of(h));
  ++h->launches;
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev_observed, h->stream));
  CU(cudaStreamWaitEvent(h->cpy, h->ev_observed, 0));
  CU(cudaMemcpyAsync(out, h->post, n * sizeof(double), cudaMemcpyDeviceToHost, h->cpy));
  CU(cudaEventRecord(h->ev_downloaded, h->cpy));
  h->download_pending = true;
  return 0;
}
}  // namespace

extern "C" {

int bflbm_stage_populations(bflbm_lattice* h, const double* f, const double* g, int ghosted) {
  CHECK_H(h);
  if (!f || !g) return fail(BFLBM_ERR_ARG, "null population buffer");
  if (ghosted != 0 && ghosted != 1) return fail(BFLBM_ERR_ARG, "ghosted must be 0 or 1");
  if (!ghosted && !h->whole_box) return fail(BFLBM_ERR_ARG, "slab lattices stage ghosted arrays (19, nz_local + 2, ny, nx)");
  if (h->pre_state) return fail(BFLBM_ERR_STATE, "a staged checkpoint is waiting for bflbm_init_from_staged");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_copy_stream(h))) return rc;
  const size_t n = (size_t)Q * (h->G.nzl + (ghosted ? 2 : 0)) * h->G.plane;  // doubles per species
  if ((rc = ensure_buffer(h, &h->pre, &h->pre_doubles, 2 * n))) return rc;
  if (h->pre_consumed_once) CU(cudaStreamWaitEvent(h->cpy, h->ev_pre_free, 0));  // the scatter of the previous checkpoint has read `pre`
  CU(cudaMemcpyAsync(h->pre, f, n * sizeof(double), cudaMemcpyHostToDevice, h->cpy));
  CU(cudaMemcpyAsync(h->pre + n, g, n * sizeof(double), cudaMemcpyHostToDevice, h->cpy));
  CU(cudaEventRecord(h->ev_staged, h->cpy));
  h->pre_state = ghosted ? 2 : 1;
  return 0;
}
int bflbm_stage_wait(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->cpy) return 0;
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaEventSynchronize(h->ev_staged));
  return 0;
}
int bflbm_init_from_staged(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->pre_state) return fail(BFLBM_ERR_STATE, "bflbm_init_from_staged: nothing staged");
  int rc = set_device(h);
  if (rc) return rc;
  const bool ghosted = h->pre_state == 2;
  const Geom& G = h->G;
  CU(cudaStreamWaitEvent(h->stream, h->ev_staged, 0));
  // the staging area holds [f | g], each (19, planes, ny, nx): the layout k_scatter_populations expects of a chunk of all planes
  k_scatter_populations<<<cell_grid(h, G.nzl + (ghosted ? 2 : 0)), h->block, 0, h->stream>>>(G, ghosted ? -1 : 0, ghosted ? 0 : 1, h->pre, h->X[h->cur]);
  ++h->launches;
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev_pre_free, h->stream));
  h->pre_consumed_once = true;
  h->pre_state = 0;
  if ((rc = finish_init(h))) return rc;
  if (h->whole_box) {
    if ((rc = bflbm_halo_refresh_begin(h))) return rc;
    return bflbm_halo_refresh_end(h);
  }
  return 0;  // a slab: the caller runs the halo refresh next, as after bflbm_init_from_populations_slab
}
int bflbm_get_hydrovars_async(bflbm_lattice* h, double* out22) { return observe_async<OBS_HYDRO>(h, BFLBM_NHYDRO, out22); }
int bflbm_get_hydrovars_bar_async(bflbm_lattice* h, double* out9) { return observe_async<OBS_HBAR>(h, BFLBM_NHYDRO_BAR, out9); }
int bflbm_download_wait(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->download_pending) return 0;
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaEventSynchronize(h->ev_downloaded));
  h->download_pending = false;
  return 0;
}
int bflbm_release_staging(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->cpy) return 0;
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->cpy));
  CU(cudaStreamSynchronize(h->stream));
  h->download_pending = false;
  h->pre_state = 0;
  h->pre_consumed_once = false;
  CU(cudaFree(h->pre));
  CU(cudaFree(h->post));
  h->bytes -= (h->pre_doubles + h->post_doubles) * sizeof(double);
  h->pre = h->post = nullptr;
  h->pre_doubles = h->post_doubles = 0;
  return 0;
}

int bflbm_params_default(bflbm_params* p) {
  if (!p) return fail(BFLBM_ERR_ARG, "null params");
  p->kBT = 0.; p->tau_f = 0.5; p->tau_g = 0.5; p->alpha0 = 4.; p->alpha1 = 0.; p->kappa = 4.;
  p->rho_lo = 0.; p->rho_hi = 1.; p->seed = 12345ull; p->step0 = 0;
  return 0;
}

int bflbm_create(const bflbm_params* p, int nx, int ny, int nz, int device, bflbm_lattice** out) {
  return create_common(p, nx, ny, nz, 0, nz, device, true, out);
}
int bflbm_create_slab(const bflbm_params* p, int nx, int ny, int nz_global, int z0, int nz_local, int device, bflbm_lattice** out) {
  return create_common(p, nx, ny, nz_global, z0, nz_local, device, false, out);
}

int bflbm_destroy(bflbm_lattice* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  drop_graphs(h);
  cudaFree(h->d_step);
  cudaFree(h->eq);
  cudaFree(h->d_shift);
  cudaFree(h->com);
  cudaFree(h->com_part);
  if (h->aux) { cudaStreamSynchronize(h->aux); cudaStreamDestroy(h->aux); }
  if (h->ev_prev) cudaEventDestroy(h->ev_prev);
  if (h->ev_ends) cudaEventDestroy(h->ev_ends);
  if (h->ev_interior) cudaEventDestroy(h->ev_interior);
  cudaFree(h->X[0]); cudaFree(h->X[1]); cudaFree(h->R); cudaFree(h->E[0]); cudaFree(h->E[1]);
  for (int s = 0; s < 2; ++s) cudaFree(h->send[s]);
  release_ipc(h);
  cudaFree(h->mailbox);
  cudaFree(h->stage); cudaFree(h->diag_partial); cudaFree(h->diag_count);
  if (h->cpy) { cudaStreamSynchronize(h->cpy); cudaStreamDestroy(h->cpy); }
  for (cudaEvent_t e : {h->ev_staged, h->ev_pre_free, h->ev_observed, h->ev_downloaded}) if (e) cudaEventDestroy(e);
  cudaFree(h->pre); cudaFree(h->post);
  for (int i = 0; i < 5; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  for (cudaEvent_t e : h->evpool) cudaEventDestroy(e);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return 0;
}

int bflbm_set_params(bflbm_lattice* h, const bflbm_params* p) {
  CHECK_H(h);
  int rc = validate_params(p);
  if (rc) return rc;
  const long long keep = h->step;
  drop_graphs(h);  // the parameters are by-value kernel arguments of the captured launches
  h->prm = *p;
  derive(h);
  h->step = h->initialized ? keep : p->step0;
  return 0;
}
int bflbm_get_params(const bflbm_lattice* h, bflbm_params* p) {
  CHECK_H(h);
  if (!p) return fail(BFLBM_ERR_ARG, "null params");
  *p = h->prm;
  return 0;
}
int bflbm_set_stream(bflbm_lattice* h, void* s) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  drop_graphs(h);
  if (h->own_stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
  if (s) h->stream = (cudaStream_t)s;
  else {
    CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;
  }
  return 0;
}
int bflbm_set_algorithm(bflbm_lattice* h, int algo) {
  CHECK_H(h);
  if (algo < 0 || algo > 1) return fail(BFLBM_ERR_ARG, "algorithm must be 0 (fused one-pass) or 1 (two-pass)");
  if (algo == 1 && !h->whole_box) return fail(BFLBM_ERR_ARG, "the two-pass algorithm supports whole-box lattices only");
  h->algo = algo;
  h->algo_auto = false;
  return bflbm_set_tiling(h, h->lz_request);  // the brick shape depends on the kernel
}

int bflbm_set_tiling(bflbm_lattice* h, int brick_lz) {
  CHECK_H(h);
  if (brick_lz < 0) return fail(BFLBM_ERR_ARG, "brick height must be >= 0");
  if (brick_lz > 0 && h->algo_auto) {  // a brick height is a request for the brick kernel
    h->algo_auto = false;
    h->algo = 0;
  }
  h->lz_request = brick_lz;
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  if (h->initialized && (rc = ensure_full_R(h))) return rc;  // E is about to change shape: R takes over
  CU(cudaStreamSynchronize(h->stream));
  h->e_valid = false;
  drop_graphs(h);
  const BrickGrid nb = make_brick_grid(h->G, brick_lz, h->cta_threads, 32);
  if (brick_doubles2(nb) != brick_doubles2(h->B)) {
    for (int k = 0; k < 2; ++k) {
      CU(cudaFree(h->E[k]));
      h->bytes -= brick_doubles2(h->B) * sizeof(double2);
      h->E[k] = nullptr;
      if ((rc = dev_alloc(h, &h->E[k], brick_doubles2(nb)))) return rc;
    }
  }
  h->B = nb;
  return 0;
}

int bflbm_init_mixture(bflbm_lattice* h) {
  CHECK_H(h);
  InitSpec S{0, h->prm.rho_lo, h->prm.rho_hi, h->prm.kappa, 0., 0.};
  return run_init(h, S);
}
int bflbm_init_stripe(bflbm_lattice* h, double frac) {
  CHECK_H(h);
  InitSpec S{1, h->prm.rho_lo, h->prm.rho_hi, h->prm.kappa, frac, 0.};
  return run_init(h, S);
}
int bflbm_init_droplet(bflbm_lattice* h, double radius) {
  CHECK_H(h);
  InitSpec S{2, h->prm.rho_lo, h->prm.rho_hi, h->prm.kappa, 0., radius};
  return run_init(h, S);
}
int bflbm_init_from_populations(bflbm_lattice* h, const double* f, const double* g) {
  CHECK_H(h);
  if (!f || !g) return fail(BFLBM_ERR_ARG, "null population buffer");
  if (!h->whole_box) return fail(BFLBM_ERR_ARG, "slab lattices need bflbm_init_from_populations_slab");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = upload_populations(h, f, g, 0))) return rc;
  // same partial-sum + self-exchange path a slab takes, so the result does not depend on the slab count
  if ((rc = finish_init(h))) return rc;
  if ((rc = bflbm_halo_refresh_begin(h))) return rc;
  return bflbm_halo_refresh_end(h);
}
int bflbm_init_from_populations_slab(bflbm_lattice* h, const double* f, const double* g) {
  CHECK_H(h);
  if (!f || !g) return fail(BFLBM_ERR_ARG, "null population buffer");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = upload_populations(h, f, g, 1))) return rc;
  if ((rc = finish_init(h))) return rc;
  // the ghost planes of X and the densities are completed by bflbm_halo_refresh_begin / exchange / _end,
  // which the caller must run next (done here for a whole box, whose neighbour is itself)
  if (h->whole_box) {
    if ((rc = bflbm_halo_refresh_begin(h))) return rc;
    return bflbm_halo_refresh_end(h);
  }
  return 0;
}

int bflbm_init_from_global_populations(bflbm_lattice* h, const double* f_global, const double* g_global) {
  CHECK_H(h);
  if (!f_global || !g_global) return fail(BFLBM_ERR_ARG, "null population buffer");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = upload_populations(h, f_global, g_global, 2))) return rc;
  if ((rc = finish_init(h))) return rc;
  // ghost planes of X and the densities: halo refresh (done here when the lattice can do it alone)
  if (h->whole_box || h->peer_mode) {
    if ((rc = bflbm_halo_refresh_begin(h))) return rc;
    if (h->whole_box) return bflbm_halo_refresh_end(h);
  }
  return 0;
}

int bflbm_set_reference_state(bflbm_lattice* h, const double* rho_eq, const double* phi_eq, const double* rhot_eq) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  drop_graphs(h);
  const Geom& G = h->G;
  const size_t n = (size_t)G.plane * G.nz_global;  // every slab holds the profiles of the whole box: the shift is unbounded
  if (!rho_eq) {  // back to the shipped behaviour: amplitudes from the current densities
    if (h->eq) {
      CU(cudaFree(h->eq));
      h->bytes -= 3 * n * sizeof(double);
    }
    h->eq = nullptr;
    h->com_pending = false;
    return 0;
  }
  if (!phi_eq || !rhot_eq) return fail(BFLBM_ERR_ARG, "null equilibrium field");
  if (!h->eq) {
    if ((rc = dev_alloc(h, &h->eq, 3 * n))) return rc;
    if (!h->d_shift && (rc = dev_alloc(h, &h->d_shift, (size_t)3))) return rc;
    if (!h->com && (rc = dev_alloc(h, &h->com, (size_t)4 * G.nz_global))) return rc;
    if (!h->com_part && (rc = dev_alloc(h, &h->com_part, (size_t)4 * G.nzl * com_chunks(G)))) return rc;
    CU(cudaMemset(h->d_shift, 0, 3 * sizeof(int)));
  }
  const double* src[3] = {rho_eq, phi_eq, rhot_eq};
  for (int k = 0; k < 3; ++k) CU(cudaMemcpy(h->eq + k * n, src[k], n * sizeof(double), cudaMemcpyHostToDevice));
  // com_ref[0] = update_com(rho_eq), main_run_job.cpp:229-233: cells of the whole box visited x fastest (the same bits on every slab)
  double m = 0., sx = 0., sy = 0., sz = 0.;
  size_t c = 0;
  for (int k = 0; k < G.nz_global; ++k)
    for (int j = 0; j < G.ny; ++j)
      for (int i = 0; i < G.nx; ++i, ++c) {
        const double r = rho_eq[c];
        m += r; sx += r * i; sy += r * j; sz += r * k;
      }
  h->com_ref[0] = sx / m; h->com_ref[1] = sy / m; h->com_ref[2] = sz / m;
  // a whole box keeps running on the thread-per-cell kernels (bflbm_set_algorithm(h, 0) moves it to the brick kernel)
  if (h->whole_box && h->algo != 1) {
    if (h->initialized && (rc = ensure_full_R(h))) return rc;
    h->algo = 1;
    h->algo_auto = false;
    h->e_valid = false;
  }
  if (h->initialized && (rc = update_ref_shift(h))) return rc;
  return 0;
}
int bflbm_get_reference_com(const bflbm_lattice* h, double* com3) {
  CHECK_H(h);
  if (!com3) return fail(BFLBM_ERR_ARG, "null output");
  if (!h->eq) return fail(BFLBM_ERR_STATE, "no reference state set");
  for (int k = 0; k < 3; ++k) com3[k] = h->com_ref[k];
  return 0;
}

size_t bflbm_com_doubles(const bflbm_lattice* h) { return h ? (size_t)4 * h->G.nz_global : 0; }
void* bflbm_com_buffer(bflbm_lattice* h) { return h ? h->com : nullptr; }
int bflbm_com_update(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->eq) return fail(BFLBM_ERR_STATE, "no reference state set");
  if (!h->com_pending) return fail(BFLBM_ERR_STATE, "no centre of mass pending (bflbm_com_update follows bflbm_step_end, an init or a restart of a slab)");
  int rc = set_device(h);
  if (rc) return rc;
  return ref_com_shift(h);
}
int bflbm_get_reference_shift(const bflbm_lattice* h, int* shift3) {
  CHECK_H(h);
  if (!shift3) return fail(BFLBM_ERR_ARG, "null output");
  if (!h->eq) return fail(BFLBM_ERR_STATE, "no reference state set");
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpy(shift3, h->d_shift, 3 * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

int bflbm_step(bflbm_lattice* h, int nsteps) {
  CHECK_H(h);
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "bflbm_step before init");
  if (!h->whole_box) return fail(BFLBM_ERR_STATE, "slab lattice: use bflbm_step_begin / exchange / bflbm_step_end");
  if (nsteps < 0) return fail(BFLBM_ERR_ARG, "nsteps < 0");
  int rc = set_device(h);
  if (rc) return rc;
  for (int s = 0; s < nsteps;) {
    if (nsteps - s >= 2 && graph_ok(h)) {
      int K = 2;
      for (int c : {64, 16, 4}) if (nsteps - s >= c) { K = c; break; }
      if ((rc = run_graph_chunk(h, K)) == 0) { s += K; continue; }
      if (h->use_graphs) return rc;  // a real failure; (capture refused -> use_graphs is off -> plain launches below)
    }
    if ((rc = step_local(h, /*pack=*/false))) return rc;
    if (h->algo == 0 && !h->wrapped_in_fold) {
      // periodic self-exchange in one launch (what pack_halo + unpack_halo of my own messages would do)
      k_wrap_whole_box<<<(unsigned)((h->G.plane + 255) / 256), 256, 0, h->stream>>>(h->G, h->X[h->cur], h->R);
      ++h->launches;
      CU(cudaGetLastError());
      if (h->eq && (rc = ref_shift_after_step(h))) return rc;
    }
    mark(h, 4);
    profile_collect(h);
    ++h->step;
    ++s;
  }
  return 0;
}
int bflbm_step_begin(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "bflbm_step_begin before init");
  if (h->algo != 0 && h->algo_auto) h->algo = 0;  // an automatically chosen two-pass whole box asked to step like a slab
  if (h->algo != 0) return fail(BFLBM_ERR_STATE, "slab stepping needs the fused algorithm");
  if (h->com_pending)
    return fail(BFLBM_ERR_STATE, "reference-state slab: the centre of mass of the last step is pending (sum all-reduce of bflbm_com_buffer "
                                 "over all slabs, then bflbm_com_update)");
  int rc = set_device(h);
  if (rc) return rc;
  return step_local(h);
}
int bflbm_step_end(bflbm_lattice* h) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  if (h->interior_pending) {  // join the interior rows before anything else touches the lattice
    CU(cudaStreamWaitEvent(h->stream, h->ev_interior, 0));
    h->interior_pending = false;
  }
  double* const self[2] = {h->send[1], h->send[0]};
  if ((rc = unpack_halo(h, h->whole_box ? self : h->recv))) return rc;
  if (h->eq && (rc = ref_shift_after_step(h))) return rc;  // a slab: its planes of the centre of mass, for the caller's all-reduce
  mark(h, 4);
  profile_collect(h);  // interval 3 (pack end -> unpack end) contains the caller's exchange (and the centre-of-mass planes)
  ++h->step;
  return 0;
}
int bflbm_halo_refresh_begin(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  h->e_valid = false;  // R is rebuilt from the populations below
  h->r_stale = false;
  // local density partials straight from the populations: P = sum over owned source planes only
  k_density_partial<<<cell_grid(h, h->G.nzl + 2), h->block, 0, h->stream>>>(h->G, h->X[h->cur], h->R);
  ++h->launches;
  CU(cudaGetLastError());
  return pack_halo(h);
}
int bflbm_halo_refresh_end(bflbm_lattice* h) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  double* const self[2] = {h->send[1], h->send[0]};
  if ((rc = unpack_halo(h, h->whole_box ? self : h->recv))) return rc;
  h->ghosts_stale = false;
  h->ref_relative = true;  // restart entry: LBM_init passes com - com_ref (LBM_binary.H:651-653)
  return update_ref_shift(h);
}
size_t bflbm_halo_doubles(const bflbm_lattice* h) { return h ? h->halo_doubles : 0; }
void* bflbm_halo_send_buffer(bflbm_lattice* h, int side) { return (h && (side == 0 || side == 1)) ? h->send[side] : nullptr; }
void* bflbm_halo_recv_buffer(bflbm_lattice* h, int side) { return (h && (side == 0 || side == 1)) ? h->recv[side] : nullptr; }

// ---- peer mode: the halo message goes straight into the neighbour's mailbox over NVLink ---------------------------------
namespace {
struct IpcOpen { void* ptr; int refs; };
std::map<std::string, IpcOpen>& ipc_table() { static std::map<std::string, IpcOpen> t; return t; }
int peer_connected(bflbm_lattice* h, int side, double* base) {
  h->peer_base[side] = base;
  h->peer_mode = h->peer_base[0] != nullptr && h->peer_base[1] != nullptr;
  return 0;
}
}  // namespace
}  // extern "C"
void release_ipc(bflbm_lattice* h) {
  auto& T = ipc_table();
  for (const std::string& k : h->ipc_keys) {
    auto it = T.find(k);
    if (it != T.end() && --it->second.refs == 0) { cudaIpcCloseMemHandle(it->second.ptr); T.erase(it); }
  }
  h->ipc_keys.clear();
}
extern "C" {
size_t bflbm_peer_mailbox_bytes(const bflbm_lattice* h) { return h ? mailbox_bytes(h) : 0; }
void* bflbm_peer_mailbox(bflbm_lattice* h) { return h ? h->mailbox : nullptr; }
int bflbm_peer_ipc_handle(bflbm_lattice* h, void* out64) {
  CHECK_H(h);
  if (!out64) return fail(BFLBM_ERR_ARG, "null output");
  static_assert(sizeof(cudaIpcMemHandle_t) == BFLBM_IPC_HANDLE_BYTES, "CUDA IPC handle size");
  int rc = set_device(h);
  if (rc) return rc;
  cudaIpcMemHandle_t hd;
  CU(cudaIpcGetMemHandle(&hd, h->mailbox));
  memcpy(out64, &hd, sizeof hd);
  return 0;
}
int bflbm_peer_connect(bflbm_lattice* h, int side, void* neighbour_mailbox, int neighbour_device) {
  CHECK_H(h);
  if (h->whole_box) return fail(BFLBM_ERR_ARG, "peer mode is for slab lattices");
  if ((side != 0 && side != 1) || !neighbour_mailbox) return fail(BFLBM_ERR_ARG, "bad side / null mailbox");
  int rc = set_device(h);
  if (rc) return rc;
  if (neighbour_device != h->device) {
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, h->device, neighbour_device));
    if (!can) return fail(BFLBM_ERR_CUDA, "device %d cannot access device %d (no NVLink / PCIe peer path)", h->device, neighbour_device);
    const cudaError_t e = cudaDeviceEnablePeerAccess(neighbour_device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(BFLBM_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
    cudaGetLastError();
  }
  return peer_connected(h, side, static_cast<double*>(neighbour_mailbox));
}
int bflbm_peer_connect_ipc(bflbm_lattice* h, int side, const void* handle64) {
  CHECK_H(h);
  if (h->whole_box) return fail(BFLBM_ERR_ARG, "peer mode is for slab lattices");
  if ((side != 0 && side != 1) || !handle64) return fail(BFLBM_ERR_ARG, "bad side / null handle");
  int rc = set_device(h);
  if (rc) return rc;
  // one mapping per (handle, device) and process: with two ranks both neighbours are the same lattice
  std::string key(static_cast<const char*>(handle64), BFLBM_IPC_HANDLE_BYTES);
  key += std::to_string(h->device);
  auto& T = ipc_table();
  auto it = T.find(key);
  if (it == T.end()) {
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle64, sizeof hd);
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
    it = T.emplace(key, IpcOpen{p, 0}).first;
  }
  ++it->second.refs;
  h->ipc_keys.push_back(key);
  return peer_connected(h, side, static_cast<double*>(it->second.ptr));
}
int bflbm_peer_connected(const bflbm_lattice* h) { return h && h->peer_mode ? 1 : 0; }
/* begin + exchange + end, nsteps times: in peer mode the exchange IS the pack kernel, so a slab steps like a whole box */
int bflbm_step_slab(bflbm_lattice* h, int nsteps) {
  CHECK_H(h);
  if (!h->peer_mode) return fail(BFLBM_ERR_STATE, "bflbm_step_slab needs both neighbours connected (bflbm_peer_connect / _ipc)");
  if (h->eq)
    return fail(BFLBM_ERR_STATE, "reference-state slab: every step needs the centre-of-mass exchange -- per step call bflbm_step_begin, "
                                 "bflbm_step_end, a sum all-reduce of bflbm_com_buffer over all slabs, bflbm_com_update");
  if (nsteps < 0) return fail(BFLBM_ERR_ARG, "nsteps < 0");
  for (int s = 0; s < nsteps; ++s) {
    int rc = bflbm_step_begin(h);
    if (rc == 0) rc = bflbm_step_end(h);
    if (rc) return rc;
  }
  return 0;
}
int bflbm_halo_refresh(bflbm_lattice* h) {
  CHECK_H(h);
  if (!h->peer_mode && !h->whole_box) return fail(BFLBM_ERR_STATE, "bflbm_halo_refresh needs peer mode (or a whole-box lattice)");
  int rc = bflbm_halo_refresh_begin(h);
  return rc ? rc : bflbm_halo_refresh_end(h);
}
int bflbm_halo_error(bflbm_lattice* h, int* flag) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  int e = 0;
  CU(cudaMemcpyAsync(&e, mailbox_err(h->mailbox, h), sizeof e, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (flag) *flag = e;
  if (e) return fail(BFLBM_ERR_STATE, "a halo wait timed out: the neighbour's message did not arrive within 10 s (rank died or call sequences differ)");
  return 0;
}

int bflbm_sync(bflbm_lattice* h) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}
long long bflbm_step_count(const bflbm_lattice* h) { return h ? h->step : -1; }
int bflbm_get_dims(const bflbm_lattice* h, int* nx, int* ny, int* nz_local, int* z0, int* nz_global) {
  CHECK_H(h);
  if (nx) *nx = h->G.nx;
  if (ny) *ny = h->G.ny;
  if (nz_local) *nz_local = h->G.nzl;
  if (z0) *z0 = h->G.z0;
  if (nz_global) *nz_global = h->G.nz_global;
  return 0;
}

int bflbm_get_populations(bflbm_lattice* h, double* f, double* g) { return observe_pair<OBS_POP>(h, f, g, false); }
int bflbm_get_populations_into_global(bflbm_lattice* h, double* f, double* g) { return observe_pair<OBS_POP>(h, f, g, true); }
int bflbm_get_populations_device(bflbm_lattice* h, double* dev_f, double* dev_g) {
  CHECK_H(h);
  if (!dev_f || !dev_g) return fail(BFLBM_ERR_ARG, "null output buffer");
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  const Geom& G = h->G;
  const int cp = chunk_planes(h, 2 * Q, 0);
  if ((rc = ensure_stage(h, (size_t)(2 * Q) * cp * G.plane))) return rc;
  for (int zlo = 0; zlo < G.nzl; zlo += cp) {
    const int zc = std::min(cp, G.nzl - zlo);
    k_observe<OBS_POP, false><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    ++h->launches;
    CU(cudaGetLastError());
    double* outs[2] = {dev_f, dev_g};
    for (int s = 0; s < 2; ++s)
      CU(cudaMemcpy2DAsync(outs[s] + (size_t)zlo * G.plane, (size_t)G.nzl * G.plane * sizeof(double), h->stage + (size_t)s * Q * zc * G.plane,
                           (size_t)zc * G.plane * sizeof(double), (size_t)zc * G.plane * sizeof(double), Q, cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  return 0;
}
int bflbm_get_hydrovars_into_global(bflbm_lattice* h, double* g22) { return observe<OBS_HYDRO>(h, BFLBM_NHYDRO, g22, false, false, true); }
int bflbm_get_hydrovars_bar_into_global(bflbm_lattice* h, double* g9) { return observe<OBS_HBAR>(h, BFLBM_NHYDRO_BAR, g9, false, false, true); }
int bflbm_get_hydrovars(bflbm_lattice* h, double* out22) { return observe<OBS_HYDRO>(h, BFLBM_NHYDRO, out22, false, false); }
int bflbm_get_hydrovars_bar(bflbm_lattice* h, double* out9) { return observe<OBS_HBAR>(h, BFLBM_NHYDRO_BAR, out9, false, false); }
int bflbm_get_hydrovars_device(bflbm_lattice* h, double* o) { return observe<OBS_HYDRO>(h, BFLBM_NHYDRO, o, true, false); }
// device array of the WHOLE box (may live on another GPU of this process: unified addressing makes the copy a peer copy)
int bflbm_get_hydrovars_device_into_global(bflbm_lattice* h, double* g22) { return observe<OBS_HYDRO>(h, BFLBM_NHYDRO, g22, true, false, true); }
int bflbm_get_device(const bflbm_lattice* h) { return h ? h->device : -1; }
int bflbm_get_hydrovars_bar_device(bflbm_lattice* h, double* o) { return observe<OBS_HBAR>(h, BFLBM_NHYDRO_BAR, o, true, false); }
int bflbm_get_noise(bflbm_lattice* h, double* fn, double* gn) { return observe_pair<OBS_NOISE>(h, fn, gn, false); }
int bflbm_get_noise_into_global(bflbm_lattice* h, double* fn, double* gn) { return observe_pair<OBS_NOISE>(h, fn, gn, true); }
int bflbm_get_normals(bflbm_lattice* h, double* out33) { return observe<OBS_NORMALS>(h, BFLBM_NNORMALS, out33, false, true); }

static int run_diag(bflbm_lattice* h, double sums[NDIAG], unsigned long long* bad) {
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  CU(cudaMemsetAsync(h->diag_count, 0, sizeof(unsigned long long), h->stream));
  k_diag<<<cell_grid(h, h->G.nzl), h->block, 0, h->stream>>>(h->G, h->R, h->diag_partial, h->diag_count);
  ++h->launches;
  CU(cudaGetLastError());
  std::vector<double> part(h->diag_blocks * NDIAG);
  CU(cudaMemcpyAsync(part.data(), h->diag_partial, part.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaMemcpyAsync(bad, h->diag_count, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int k = 0; k < NDIAG; ++k) sums[k] = 0.;
  for (size_t b = 0; b < h->diag_blocks; ++b)
    for (int k = 0; k < NDIAG; ++k) sums[k] += part[b * NDIAG + k];
  return 0;
}
int bflbm_center_of_mass(bflbm_lattice* h, double* com3, double* sums4) {
  CHECK_H(h);
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  double s[NDIAG];
  unsigned long long bad;
  int rc = run_diag(h, s, &bad);
  if (rc) return rc;
  if (com3) { com3[0] = s[2] / s[0]; com3[1] = s[3] / s[0]; com3[2] = s[4] / s[0]; }
  if (sums4) { sums4[0] = s[0]; sums4[1] = s[2]; sums4[2] = s[3]; sums4[3] = s[4]; }
  return 0;
}
int bflbm_total_mass(bflbm_lattice* h, double* mr, double* mp) {
  CHECK_H(h);
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  double s[NDIAG];
  unsigned long long bad;
  int rc = run_diag(h, s, &bad);
  if (rc) return rc;
  if (mr) *mr = s[0];
  if (mp) *mp = s[1];
  return 0;
}
int bflbm_second_moments(bflbm_lattice* h, double* sums10) {
  CHECK_H(h);
  if (!sums10) return fail(BFLBM_ERR_ARG, "null output");
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  double s[NDIAG];
  unsigned long long bad;
  int rc = run_diag(h, s, &bad);
  if (rc) return rc;
  sums10[0] = s[0];
  for (int k = 1; k < 10; ++k) sums10[k] = s[k + 1];
  return 0;
}
// eigenvalues of a symmetric 3x3 matrix {xx, yy, zz, xy, xz, yz}, ascending (trigonometric closed form)
static void sym3_eigenvalues(const double c[6], double e[3]) {
  const double p1 = c[3] * c[3] + c[4] * c[4] + c[5] * c[5];
  const double q = (c[0] + c[1] + c[2]) / 3.;
  const double p2 = (c[0] - q) * (c[0] - q) + (c[1] - q) * (c[1] - q) + (c[2] - q) * (c[2] - q) + 2. * p1;
  if (p2 <= 0.) { e[0] = e[1] = e[2] = q; return; }
  const double p = sqrt(p2 / 6.);
  const double b[6] = {(c[0] - q) / p, (c[1] - q) / p, (c[2] - q) / p, c[3] / p, c[4] / p, c[5] / p};
  const double det = b[0] * (b[1] * b[2] - b[5] * b[5]) - b[3] * (b[3] * b[2] - b[5] * b[4]) + b[4] * (b[3] * b[5] - b[1] * b[4]);
  const double r = std::max(-1., std::min(1., det / 2.));
  const double phi = acos(r) / 3.;
  e[2] = q + 2. * p * cos(phi);
  e[0] = q + 2. * p * cos(phi + 2. * M_PI / 3.);
  e[1] = 3. * q - e[0] - e[2];
}
// centre of mass, mass-weighted covariance and its eigenvalues from the ten sums {M, Mx, My, Mz, Mxx, Myy, Mzz, Mxy, Mxz, Myz}
// (pure host arithmetic: lets the caller combine bflbm_second_moments of several slabs first)
int bflbm_covariance_from_moments(const double* m, double* com3, double* cov6, double* eig3) {
  if (!m) return fail(BFLBM_ERR_ARG, "null sums");
  const double M = m[0], cx = m[1] / M, cy = m[2] / M, cz = m[3] / M;
  const double c[6] = {m[4] / M - cx * cx, m[5] / M - cy * cy, m[6] / M - cz * cz, m[7] / M - cx * cy, m[8] / M - cx * cz, m[9] / M - cy * cz};
  if (com3) { com3[0] = cx; com3[1] = cy; com3[2] = cz; }
  if (cov6) for (int k = 0; k < 6; ++k) cov6[k] = c[k];
  if (eig3) sym3_eigenvalues(c, eig3);
  return 0;
}
int bflbm_droplet_covariance(bflbm_lattice* h, double* com3, double* cov6, double* eig3) {
  CHECK_H(h);
  if (!h->whole_box) return fail(BFLBM_ERR_ARG, "slab lattice: combine bflbm_second_moments of all slabs (bflbm_covariance_from_moments) or use bflbm_multi");
  double m[10];
  int rc = bflbm_second_moments(h, m);
  if (rc) return rc;
  return bflbm_covariance_from_moments(m, com3, cov6, eig3);
}
// ---- droplet (W, R) fit, SURVEY 8(f) row 4 (droplet_fit.hpp) ---------------------------------------------------------------------
// local partial sums over this lattice's cells: sums4 = {sum rho (R - r') sech^2, sum rho sech^2, min rho, max rho}
int bflbm_droplet_fit_terms(bflbm_lattice* h, double W, double Rn, const double* r0, double* sums4) {
  CHECK_H(h);
  if (!r0 || !sums4) return fail(BFLBM_ERR_ARG, "null argument");
  if (!(W > 0.)) return fail(BFLBM_ERR_ARG, "W must be > 0");
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  k_fit_terms<<<cell_grid(h, h->G.nzl), h->block, 0, h->stream>>>(h->G, h->R, 1. / sqrt(2. * W), Rn, r0[0], r0[1], r0[2], h->diag_partial);
  ++h->launches;
  CU(cudaGetLastError());
  static_assert(NDIAG >= 4, "the diagnostics buffer holds at least four values per block");
  std::vector<double> part(h->diag_blocks * 4);
  CU(cudaMemcpyAsync(part.data(), h->diag_partial, part.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  sums4[0] = sums4[1] = 0.;
  sums4[2] = 1e300;
  sums4[3] = -1e300;
  for (size_t b = 0; b < h->diag_blocks; ++b) {  // block order: the same sum on every run
    sums4[0] += part[b * 4];
    sums4[1] += part[b * 4 + 1];
    sums4[2] = std::min(sums4[2], part[b * 4 + 2]);
    sums4[3] = std::max(sums4[3], part[b * 4 + 3]);
  }
  return 0;
}
int bflbm_fit_droplet(bflbm_lattice* h, int step_window, double undul_ratio, int nstep, double W0, double R0, double eta_W, double eta_R,
                      double dt, double* out3, int* converged) {
  CHECK_H(h);
  if (!out3) return fail(BFLBM_ERR_ARG, "null output");
  if (!h->whole_box) return fail(BFLBM_ERR_ARG, "slab lattice: use bflbm_multi_fit_droplet (or combine bflbm_droplet_fit_terms of all slabs)");
  if (nstep < 2 || step_window < 1 || step_window > nstep || !(W0 > 0.)) return fail(BFLBM_ERR_ARG, "bad fit parameters");
  double com[3];
  int rc = bflbm_center_of_mass(h, com, nullptr);  // cell indices; cell centres in the unit cube: (i + 1/2) / n (LBM_hydrovs.H:92-96)
  if (rc) return rc;
  const double r0[3] = {(com[0] + 0.5) / h->G.nx, (com[1] + 0.5) / h->G.ny, (com[2] + 0.5) / h->G.nz_global};
  double s4[4];
  if ((rc = bflbm_droplet_fit_terms(h, W0, R0, r0, s4))) return rc;
  const double range = s4[3] - s4[2];
  fit::FieldTerms terms = [h](double W, double R, const double* c, double* sums) {
    double t[4];
    const int e = bflbm_droplet_fit_terms(h, W, R, c, t);
    sums[0] = t[0];
    sums[1] = t[1];
    return e;
  };
  fit::Result res;
  const double vol = 1. / ((double)h->G.nx * h->G.ny * h->G.nz_global);
  if ((rc = fit::fit(terms, vol, r0, range, step_window, undul_ratio, nstep, W0, R0, eta_W, eta_R, dt, res))) return rc;
  out3[0] = res.W; out3[1] = res.R; out3[2] = res.undulation;
  if (converged) *converged = res.converged ? 1 : 0;
  return 0;
}
// the closed-form coefficients of one flow step (test hook: pure host arithmetic, runs without a GPU)
int bflbm_debug_fit_coefficients(double W, double R, double eta_W, double eta_R, double dt, double C0, double* out6) {
  if (!out6 || !(W > 0.)) return fail(BFLBM_ERR_ARG, "bad argument");
  const fit::Coefficients q = fit::coefficients(W, R, eta_W, eta_R, dt, C0, fit::sech4_coefficients(fit::SERIES_TERMS));
  out6[0] = q.JRR; out6[1] = q.JWR; out6[2] = q.JRW; out6[3] = q.JWW; out6[4] = q.KW; out6[5] = q.KR;
  return 0;
}

int bflbm_check_nan(bflbm_lattice* h, long long* count) {
  CHECK_H(h);
  if (!h->initialized) return fail(BFLBM_ERR_STATE, "lattice not initialised");
  int rc = set_device(h);
  if (rc) return rc;
  if ((rc = ensure_full_R(h))) return rc;
  const Geom& G = h->G;
  const bool noise = h->prm.kBT > 0.;
  const int cp = chunk_planes(h, BFLBM_NHYDRO, 0);
  if ((rc = ensure_stage(h, (size_t)BFLBM_NHYDRO * cp * G.plane))) return rc;
  CU(cudaMemsetAsync(h->diag_count, 0, sizeof(unsigned long long), h->stream));
  for (int zlo = 0; zlo < G.nzl; zlo += cp) {
    const int zc = std::min(cp, G.nzl - zlo);
    if (noise) k_observe<OBS_HYDRO, true><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    else       k_observe<OBS_HYDRO, false><<<cell_grid(h, zc), h->block, 0, h->stream>>>(G, h->dp, h->step, zlo, h->X[h->cur], h->R, h->stage, rs_of(h));
    const long long n = (long long)BFLBM_NHYDRO * zc * G.plane;
    k_count_nonfinite<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->stage, n, h->diag_count);
    h->launches += 2;
    CU(cudaGetLastError());
  }
  unsigned long long bad = 0;
  CU(cudaMemcpyAsync(&bad, h->diag_count, sizeof bad, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (count) *count = (long long)bad;
  if (bad) return fail(BFLBM_ERR_NAN, "%llu non-finite values in the hydrodynamic fields at step %lld", bad, h->step);
  return 0;
}

int bflbm_set_profiling(bflbm_lattice* h, int on) {
  CHECK_H(h);
  int rc = set_device(h);
  if (rc) return rc;
  if (on < 0 || on > 2) return fail(BFLBM_ERR_ARG, "profiling mode must be 0 (off), 1 (read back every step) or 2 (deferred)");
  if (on && !h->ev[0])
    for (int i = 0; i < 5; ++i) CU(cudaEventCreate(&h->ev[i]));
  if (on == 2 && h->evpool.empty()) {
    h->evpool.resize((size_t)bflbm_lattice::PROF_POOL_STEPS * 5, nullptr);
    for (cudaEvent_t& e : h->evpool) CU(cudaEventCreate(&e));
  }
  h->profiling = on != 0;
  h->prof_deferred = on == 2;
  h->prof_slot = 0;
  for (int i = 0; i < 4; ++i) h->prof_ms[i] = 0.;
  h->prof_steps = 0;
  return 0;
}
int bflbm_get_profile(bflbm_lattice* h, double ms4[4], long long* steps) {
  CHECK_H(h);
  if (!ms4) return fail(BFLBM_ERR_ARG, "null output");
  if (h->prof_deferred) {
    int rc = set_device(h);
    if (rc) return rc;
    profile_flush(h);
  }
  for (int i = 0; i < 4; ++i) ms4[i] = h->prof_ms[i];
  if (steps) *steps = h->prof_steps;
  return 0;
}

long long bflbm_kernel_launches(const bflbm_lattice* h) { return h ? h->launches : 0; }
size_t bflbm_device_bytes(const bflbm_lattice* h) { return h ? h->bytes : 0; }

int bflbm_debug_philox(const unsigned int ctr[4], const unsigned int key[2], unsigned int out[4]) {
  if (!ctr || !key || !out) return fail(BFLBM_ERR_ARG, "null argument");
  uint4* d = nullptr;
  CU(cudaMalloc((void**)&d, sizeof(uint4)));
  k_philox_test<<<1, 1>>>(make_uint4(ctr[0], ctr[1], ctr[2], ctr[3]), make_uint2(key[0], key[1]), d);
  uint4 r;
  cudaError_t e = cudaMemcpy(&r, d, sizeof r, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(BFLBM_ERR_CUDA, "philox test: %s", cudaGetErrorString(e));
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
  return 0;
}

int bflbm_debug_last_step(const bflbm_lattice* h, int out[BFLBM_LAST_STEP_FIELDS]) {
  CHECK_H(h);
  if (!out) return fail(BFLBM_ERR_ARG, "null output");
  if (!h->last_step_set) return fail(BFLBM_ERR_STATE, "no step has been launched yet");
  std::copy(h->last_step.begin(), h->last_step.end(), out);
  return 0;
}

int bflbm_debug_normal_statistics(unsigned long long seed, long long ncells, long long step0, int nsteps, int nbins, double lo, double hi,
                                  unsigned long long* hist, unsigned long long* joint, double* moments4) {
  if (!hist || !joint || !moments4 || ncells < 1 || nsteps < 1 || nbins < 1 || nbins > 4096 || !(hi > lo)) return fail(BFLBM_ERR_ARG, "bad argument");
  // a thread adds at most 33 * nsteps * (cells per thread) to one 32-bit shared counter per launch: bound the work per launch
  const size_t nh = (size_t)nbins + 2, nj = (size_t)NORMAL_JOINT_BINS * NORMAL_JOINT_BINS;
  unsigned long long *dh = nullptr, *dj = nullptr;
  double* dm = nullptr;
  CU(cudaMalloc((void**)&dh, nh * sizeof(unsigned long long)));
  CU(cudaMalloc((void**)&dj, nj * sizeof(unsigned long long)));
  CU(cudaMalloc((void**)&dm, 4 * sizeof(double)));
  CU(cudaMemset(dh, 0, nh * sizeof(unsigned long long)));
  CU(cudaMemset(dj, 0, nj * sizeof(unsigned long long)));
  CU(cudaMemset(dm, 0, 4 * sizeof(double)));
  const PhiloxKeys K = philox_key_schedule(seed);
  const size_t smem = (nh + nj) * sizeof(unsigned int);
  // per launch: 148 * 8 CTAs x 256 threads, each thread <= 16 cells x <= 64 steps x 33 draws = 33 792 increments (< 2^32 per CTA counter)
  const long long chunk_cells = 148ll * 8 * 256 * 16;
  for (long long c0 = 0; c0 < ncells; c0 += chunk_cells)
    for (int s0 = 0; s0 < nsteps; s0 += 64) {
      const long long nc = std::min(chunk_cells, ncells - c0);
      k_normal_stats<<<148 * 8, 256, smem>>>(K, nc, step0 + s0 + (c0 << 20), std::min(64, nsteps - s0), nbins, lo, hi, dh, dj, dm);
      CU(cudaGetLastError());
    }
  // (cells of later chunks are decorrelated from earlier ones through the step word of the counter instead of the cell word:
  //  the kernel numbers its cells from 0)
  CU(cudaMemcpy(hist, dh, nh * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(joint, dj, nj * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(moments4, dm, 4 * sizeof(double), cudaMemcpyDeviceToHost));
  cudaFree(dh); cudaFree(dj); cudaFree(dm);
  return 0;
}

const char* bflbm_last_error(void) { return g_err.c_str(); }
const char* bflbm_version(void) { return "bflbm-b200 0.1 (sm_100a, fp64, D3Q19 binary fluctuating)"; }

}  // extern "C"
