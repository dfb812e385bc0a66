// bflbm_multi: one periodic box on several GPUs of ONE process (include/bflbm.h, "one box on several GPUs").
//
// The reference decomposes its domain with BoxArray::maxSize + DistributionMapping and lets FillBoundary move ghost cells
// between MPI ranks (main_run_job.cpp:140-145, LBM_binary.H:553-555).  Here the box is cut into z-slabs, one per device,
// the slabs are connected in a periodic ring through their peer-mapped mailboxes (capi.cu, "peer mode"), and a step is
//     for every slab: bflbm_step_begin   (end brick rows, slab-face fold, pack kernel = the NVLink transfer;
//                                         interior rows on the slab's second stream)
//     for every slab: bflbm_step_end     (device-side wait on the arrival flags, unpack)
// -- no NCCL, no MPI, no host synchronisation: the host thread only queues launches.  With one device the object is a
// plain whole-box lattice (CUDA-graph replay for the small boxes).  Everything here goes through the public C ABI.
//
// Reference-state noise on slabs (bflbm_multi_set_reference_state): after every bflbm_step_end (and init) each slab holds the
// per-plane centre-of-mass sums of its own planes in its bflbm_com_buffer; the sum all-reduce the ABI asks for is done here with
// peer copies of each slab's planes into every other slab's buffer, ordered by cross-device events on per-slab streams that
// this object owns, then bflbm_com_update.  Still no host synchronisation in the step loop.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <new>
#include <string>
#include <vector>

#include "../../include/bflbm.h"
#include "droplet_fit.hpp"

struct bflbm_multi {
  std::vector<bflbm_lattice*> L;
  std::vector<int> dev, z0, nzl;
  int nx = 0, ny = 0, nz = 0;
  bool whole = true;
  // reference-state noise on slabs: per-slab streams (handed to the lattices) and events of the centre-of-mass exchange
  bool ref = false, initialized = false, copies_in_flight = false;
  std::vector<cudaStream_t> st;
  std::vector<cudaEvent_t> ev_com, ev_copied;
};

namespace {
thread_local std::string g_merr;
int mfail(int code, const std::string& msg) {
  g_merr = msg;
  return code;
}
#define MCHECK(m) \
  if (!(m)) return mfail(BFLBM_ERR_ARG, "null bflbm_multi handle")
// run `call` on every slab, stop at the first failure
#define FOR_ALL(m, call)                                   \
  do {                                                     \
    for (bflbm_lattice * l : (m)->L) {                     \
      const int rc_ = (call);                              \
      if (rc_) return mfail(rc_, bflbm_last_error());      \
    }                                                      \
  } while (0)
}  // namespace

extern "C" {

const char* bflbm_multi_last_error(void) { return g_merr.c_str(); }

int bflbm_multi_destroy(bflbm_multi* m) {
  if (!m) return 0;
  for (bflbm_lattice* l : m->L) bflbm_destroy(l);  // synchronises each lattice's stream first
  for (size_t r = 0; r < m->st.size(); ++r) {
    cudaSetDevice(m->dev[r]);
    cudaEventDestroy(m->ev_com[r]);
    cudaEventDestroy(m->ev_copied[r]);
    cudaStreamDestroy(m->st[r]);
  }
  delete m;
  return 0;
}

namespace {
#define MCU(call)                                                                                   \
  do {                                                                                              \
    const cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) return mfail(BFLBM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)
// a slab may overwrite its centre-of-mass buffer (bflbm_step_end, inits) only after every other slab has copied its planes
int wait_com_copies(bflbm_multi* m) {
  if (!m->copies_in_flight) return 0;
  const int P = (int)m->L.size();
  for (int s = 0; s < P; ++s) {
    MCU(cudaSetDevice(m->dev[s]));
    for (int r = 0; r < P; ++r)
      if (r != s) MCU(cudaStreamWaitEvent(m->st[s], m->ev_copied[r], 0));
  }
  m->copies_in_flight = false;
  return 0;
}
// the sum all-reduce of bflbm_com_buffer: slab s's planes [z0_s, z0_s + nzl_s) are its own, everything else is zero, so the sum is
// a copy of each owner's planes
int exchange_com(bflbm_multi* m) {
  const int P = (int)m->L.size();
  for (int r = 0; r < P; ++r) {
    MCU(cudaSetDevice(m->dev[r]));
    MCU(cudaEventRecord(m->ev_com[r], m->st[r]));
  }
  for (int r = 0; r < P; ++r) {
    MCU(cudaSetDevice(m->dev[r]));
    double* dst = static_cast<double*>(bflbm_com_buffer(m->L[r]));
    for (int s = 0; s < P; ++s) {
      if (s == r) continue;
      const double* src = static_cast<const double*>(bflbm_com_buffer(m->L[s]));
      MCU(cudaStreamWaitEvent(m->st[r], m->ev_com[s], 0));
      MCU(cudaMemcpyPeerAsync(dst + 4 * (size_t)m->z0[s], m->dev[r], src + 4 * (size_t)m->z0[s], m->dev[s], 4 * (size_t)m->nzl[s] * sizeof(double),
                              m->st[r]));
    }
    const int rc = bflbm_com_update(m->L[r]);
    if (rc) return mfail(rc, bflbm_last_error());
    MCU(cudaEventRecord(m->ev_copied[r], m->st[r]));
  }
  m->copies_in_flight = true;
  return 0;
}
// after an init: the slabs' centre of mass
int after_init(bflbm_multi* m) {
  m->initialized = true;
  return (m->ref && !m->whole) ? exchange_com(m) : 0;
}
}  // namespace

int bflbm_multi_set_reference_state(bflbm_multi* m, const double* rho_eq, const double* phi_eq, const double* rhot_eq) {
  MCHECK(m);
  if (!m->whole && rho_eq && m->st.empty()) {
    for (size_t r = 0; r < m->L.size(); ++r) {
      MCU(cudaSetDevice(m->dev[r]));
      cudaStream_t s = nullptr;
      cudaEvent_t a = nullptr, b = nullptr;
      cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&a, cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b, cudaEventDisableTiming);
      if (e != cudaSuccess) {  // the three vectors only ever hold complete triples (bflbm_multi_destroy walks them together)
        if (b) cudaEventDestroy(b);
        if (a) cudaEventDestroy(a);
        if (s) cudaStreamDestroy(s);
        return mfail(BFLBM_ERR_CUDA, std::string("centre-of-mass stream / events: ") + cudaGetErrorString(e));
      }
      m->st.push_back(s);
      m->ev_com.push_back(a);
      m->ev_copied.push_back(b);
      const int rc = bflbm_set_stream(m->L[r], s);
      if (rc) return mfail(rc, bflbm_last_error());
    }
  }
  if (int rc = wait_com_copies(m)) return rc;
  FOR_ALL(m, bflbm_set_reference_state(l, rho_eq, phi_eq, rhot_eq));
  m->ref = rho_eq != nullptr;
  return (m->ref && m->initialized && !m->whole) ? exchange_com(m) : 0;
}

int bflbm_multi_create(const bflbm_params* p, int nx, int ny, int nz, int ngpus, const int* devices, int brick_lz, bflbm_multi** out) {
  if (!out) return mfail(BFLBM_ERR_ARG, "null out pointer");
  *out = nullptr;
  if (ngpus < 1) return mfail(BFLBM_ERR_ARG, "ngpus must be >= 1");
  if (ngpus > 1 && nz / ngpus < 2) return mfail(BFLBM_ERR_ARG, "nz is too small for this many slabs (need >= 2 planes per slab)");
  bflbm_multi* m = new (std::nothrow) bflbm_multi;
  if (!m) return mfail(BFLBM_ERR_ARG, "out of host memory");
  m->nx = nx; m->ny = ny; m->nz = nz;
  m->whole = ngpus == 1;
  int rc = 0;
  for (int r = 0; r < ngpus && !rc; ++r) {
    // contiguous slabs, sizes differ by at most one plane (remainder to the low ranks)
    const int base = nz / ngpus, rem = nz % ngpus;
    const int nzl = base + (r < rem ? 1 : 0), z0 = r * base + (r < rem ? r : rem);
    const int d = devices ? devices[r] : r;
    bflbm_lattice* l = nullptr;
    rc = m->whole ? bflbm_create(p, nx, ny, nz, d, &l) : bflbm_create_slab(p, nx, ny, nz, z0, nzl, d, &l);
    if (rc) break;
    m->L.push_back(l);
    m->dev.push_back(d);
    m->z0.push_back(z0);
    m->nzl.push_back(nzl);
    if (brick_lz > 0) rc = bflbm_set_tiling(l, brick_lz);
  }
  for (int r = 0; r < ngpus && !rc && !m->whole; ++r) {
    const int lo = (r + ngpus - 1) % ngpus, hi = (r + 1) % ngpus;
    rc = bflbm_peer_connect(m->L[r], 0, bflbm_peer_mailbox(m->L[lo]), m->dev[lo]);
    if (!rc) rc = bflbm_peer_connect(m->L[r], 1, bflbm_peer_mailbox(m->L[hi]), m->dev[hi]);
  }
  if (rc) {
    mfail(rc, bflbm_last_error());
    bflbm_multi_destroy(m);
    return rc;
  }
  *out = m;
  return 0;
}

int bflbm_multi_count(const bflbm_multi* m) { return m ? (int)m->L.size() : 0; }
bflbm_lattice* bflbm_multi_slab(bflbm_multi* m, int i) { return (m && i >= 0 && i < (int)m->L.size()) ? m->L[i] : nullptr; }

int bflbm_multi_set_params(bflbm_multi* m, const bflbm_params* p) { MCHECK(m); FOR_ALL(m, bflbm_set_params(l, p)); return 0; }
#define MULTI_INIT(call)                          \
  do {                                            \
    MCHECK(m);                                    \
    if (int rc_ = wait_com_copies(m)) return rc_; \
    FOR_ALL(m, call);                             \
    return after_init(m);                         \
  } while (0)
int bflbm_multi_init_mixture(bflbm_multi* m) { MULTI_INIT(bflbm_init_mixture(l)); }
int bflbm_multi_init_stripe(bflbm_multi* m, double frac) { MULTI_INIT(bflbm_init_stripe(l, frac)); }
int bflbm_multi_init_droplet(bflbm_multi* m, double radius) { MULTI_INIT(bflbm_init_droplet(l, radius)); }
#undef MULTI_INIT
int bflbm_multi_init_from_populations(bflbm_multi* m, const double* f, const double* g) {
  MCHECK(m);
  if (int rc = wait_com_copies(m)) return rc;
  // every slab uploads its planes (+ the periodic neighbour planes) and packs its halo message; then all of them unpack
  FOR_ALL(m, bflbm_init_from_global_populations(l, f, g));
  if (!m->whole) FOR_ALL(m, bflbm_halo_refresh_end(l));
  return after_init(m);
}

int bflbm_multi_step(bflbm_multi* m, int nsteps) {
  MCHECK(m);
  if (nsteps < 0) return mfail(BFLBM_ERR_ARG, "nsteps < 0");
  if (m->whole) {
    FOR_ALL(m, bflbm_step(l, nsteps));
    return 0;
  }
  for (int s = 0; s < nsteps; ++s) {
    FOR_ALL(m, bflbm_step_begin(l));
    if (int rc = wait_com_copies(m)) return rc;  // bflbm_step_end writes the centre-of-mass planes
    FOR_ALL(m, bflbm_step_end(l));
    if (m->ref)
      if (int rc = exchange_com(m)) return rc;
  }
  return 0;
}
int bflbm_multi_sync(bflbm_multi* m) { MCHECK(m); FOR_ALL(m, bflbm_sync(l)); return 0; }
long long bflbm_multi_step_count(const bflbm_multi* m) { return (m && !m->L.empty()) ? bflbm_step_count(m->L[0]) : -1; }

int bflbm_multi_get_populations(bflbm_multi* m, double* f, double* g) { MCHECK(m); FOR_ALL(m, bflbm_get_populations_into_global(l, f, g)); return 0; }
int bflbm_multi_get_hydrovars(bflbm_multi* m, double* out22) { MCHECK(m); FOR_ALL(m, bflbm_get_hydrovars_into_global(l, out22)); return 0; }
int bflbm_multi_get_hydrovars_bar(bflbm_multi* m, double* out9) { MCHECK(m); FOR_ALL(m, bflbm_get_hydrovars_bar_into_global(l, out9)); return 0; }
int bflbm_multi_get_noise(bflbm_multi* m, double* fn, double* gn) { MCHECK(m); FOR_ALL(m, bflbm_get_noise_into_global(l, fn, gn)); return 0; }

int bflbm_multi_second_moments(bflbm_multi* m, double* sums10) {
  MCHECK(m);
  if (!sums10) return mfail(BFLBM_ERR_ARG, "null output");
  for (int k = 0; k < 10; ++k) sums10[k] = 0.;
  for (bflbm_lattice* l : m->L) {  // slab order: the same partial sums in the same order on every run
    double s[10];
    const int rc = bflbm_second_moments(l, s);
    if (rc) return mfail(rc, bflbm_last_error());
    for (int k = 0; k < 10; ++k) sums10[k] += s[k];
  }
  return 0;
}
int bflbm_multi_total_mass(bflbm_multi* m, double* mass_rho, double* mass_phi) {
  MCHECK(m);
  double a = 0., b = 0.;
  for (bflbm_lattice* l : m->L) {
    double r = 0., p = 0.;
    const int rc = bflbm_total_mass(l, &r, &p);
    if (rc) return mfail(rc, bflbm_last_error());
    a += r; b += p;
  }
  if (mass_rho) *mass_rho = a;
  if (mass_phi) *mass_phi = b;
  return 0;
}
int bflbm_multi_droplet_covariance(bflbm_multi* m, double* com3, double* cov6, double* eig3) {
  double s[10];
  const int rc = bflbm_multi_second_moments(m, s);
  if (rc) return rc;
  return bflbm_covariance_from_moments(s, com3, cov6, eig3);
}
int bflbm_multi_center_of_mass(bflbm_multi* m, double* com3) { return bflbm_multi_droplet_covariance(m, com3, nullptr, nullptr); }

// fittingDropletParams over all slabs: every flow step sums the slabs' field terms (bflbm_droplet_fit_terms)
int bflbm_multi_fit_droplet(bflbm_multi* m, int step_window, double undul_ratio, int nstep, double W0, double R0, double eta_W, double eta_R,
                            double dt, double* out3, int* converged) {
  MCHECK(m);
  if (!out3) return mfail(BFLBM_ERR_ARG, "null output");
  if (m->whole) {
    const int rc = bflbm_fit_droplet(m->L[0], step_window, undul_ratio, nstep, W0, R0, eta_W, eta_R, dt, out3, converged);
    return rc ? mfail(rc, bflbm_last_error()) : 0;
  }
  if (nstep < 2 || step_window < 1 || step_window > nstep || !(W0 > 0.)) return mfail(BFLBM_ERR_ARG, "bad fit parameters");
  double com[3];
  int rc = bflbm_multi_center_of_mass(m, com);
  if (rc) return rc;
  const double r0[3] = {(com[0] + 0.5) / m->nx, (com[1] + 0.5) / m->ny, (com[2] + 0.5) / m->nz};
  auto all = [m](double W, double R, const double* c, double* s4) {
    s4[0] = s4[1] = 0.; s4[2] = 1e300; s4[3] = -1e300;
    for (bflbm_lattice* l : m->L) {
      double t[4];
      const int e = bflbm_droplet_fit_terms(l, W, R, c, t);
      if (e) return e;
      s4[0] += t[0]; s4[1] += t[1]; s4[2] = std::min(s4[2], t[2]); s4[3] = std::max(s4[3], t[3]);
    }
    return 0;
  };
  double s4[4];
  if ((rc = all(W0, R0, r0, s4))) return mfail(rc, bflbm_last_error());
  const double range = s4[3] - s4[2];
  bflbm::fit::FieldTerms terms = [&all](double W, double R, const double* c, double* sums) {
    double t[4];
    const int e = all(W, R, c, t);
    sums[0] = t[0]; sums[1] = t[1];
    return e;
  };
  bflbm::fit::Result res;
  if ((rc = bflbm::fit::fit(terms, 1. / ((double)m->nx * m->ny * m->nz), r0, range, step_window, undul_ratio, nstep, W0, R0, eta_W, eta_R, dt, res)))
    return mfail(rc, bflbm_last_error());
  out3[0] = res.W; out3[1] = res.R; out3[2] = res.undulation;
  if (converged) *converged = res.converged ? 1 : 0;
  return 0;
}

int bflbm_multi_check_nan(bflbm_multi* m, long long* count) {
  MCHECK(m);
  long long tot = 0;
  int worst = 0;
  for (bflbm_lattice* l : m->L) {
    long long c = 0;
    const int rc = bflbm_check_nan(l, &c);
    if (rc && rc != BFLBM_ERR_NAN) return mfail(rc, bflbm_last_error());
    if (rc) { worst = rc; mfail(rc, bflbm_last_error()); }
    tot += c;
    if (!m->whole) {
      const int re = bflbm_halo_error(l, nullptr);
      if (re) return mfail(re, bflbm_last_error());
    }
  }
  if (count) *count = tot;
  return worst;
}
long long bflbm_multi_kernel_launches(const bflbm_multi* m) {
  long long n = 0;
  if (m) for (bflbm_lattice* l : m->L) n += bflbm_kernel_launches(l);
  return n;
}
size_t bflbm_multi_device_bytes(const bflbm_multi* m) {
  size_t n = 0;
  if (m) for (bflbm_lattice* l : m->L) n += bflbm_device_bytes(l);
  return n;
}

}  // extern "C"
