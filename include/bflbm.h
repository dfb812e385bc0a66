/* bflbm.h -- C ABI of the B200-native fluctuating binary D3Q19 lattice-Boltzmann step.
 *
 * This is the drop-in boundary for ONE hot path of MDProject/Binary-Fluctuating-Lattice-Boltzmann:
 * the per-step update in LBM_binary.H / LBM_d3q19.H.  The reference has no FFI; its boundary is a
 * set of header-inline C++ functions on caller-owned amrex::MultiFab objects plus global parameters.
 * Each entry point below names the reference interface it replaces (file:line in the reference).
 *
 * Conventions
 *  - Device memory is owned by the library; host buffers by the caller.
 *  - Host arrays are float64 in AMReX FAB order for the VALID region: x fastest, then y, z,
 *    component slowest, i.e. C shape (ncomp, nz_local, ny, nx).
 *  - Every call returns 0 on success or a negative bflbm_status; bflbm_last_error() gives the text.
 *    The library never calls exit() (the reference's NaN check does: Debug.H:137-149).
 *  - A lattice may be the whole periodic box (bflbm_create) or one z-slab of it (bflbm_create_slab);
 *    slabs exchange one ghost message per step through the bflbm_halo_* calls.
 *  - "time" convention (SURVEY.md section 9, item 9): after n calls of the reference's LBM_timestep
 *    the MultiFabs hold post-stream populations of time n and hydrovs/noise derived from them;
 *    all bflbm_get_* calls return exactly those quantities after n steps.
 *  - There is no CPU fallback: every entry point fails with BFLBM_ERR_CUDA if no sm_100 device
 *    can be used.
 */
#ifndef BFLBM_H_
#define BFLBM_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BFLBM_NVEL 19      /* LBM_d3q19.H:4 */
#define BFLBM_NHYDRO 22    /* main_run_job.cpp:147, names in AMReX_FileIO.H:208-261 */
#define BFLBM_NHYDRO_BAR 9 /* components of hydrovsbar that are ever written: LBM_binary.H:329-339 */
#define BFLBM_NNORMALS 33  /* Gaussian draws per cell per step: LBM_binary.H:115-127 */

typedef enum {
  BFLBM_OK = 0,
  BFLBM_ERR_ARG = -1,    /* bad argument / unsupported parameter (e.g. alpha1 != 0, use_SC_pseudo) */
  BFLBM_ERR_CUDA = -2,   /* CUDA runtime error or no usable device */
  BFLBM_ERR_STATE = -3,  /* call order (e.g. step before init) */
  BFLBM_ERR_NAN = -4     /* returned by bflbm_check_nan when a NaN/Inf is present */
} bflbm_status;

/* Every tunable the reference exposes by editing source.
 * kBT: LBM_d3q19.H:10.  seed, tau_f, tau_g, alpha0, alpha1, rho_lo, rho_hi, kappa: LBM_binary.H:17-30.
 * alpha1 does not enter the dynamics in the reference (LBM_binary.H:256-257 commented out); must be 0.
 * step0: value of the step counter at creation (main_run_job.cpp:80 step_continue); the noise is a
 *        pure function of (seed, global cell, step, draw) so a restart with the same step0 continues
 *        the same random sequence (the reference does not checkpoint its RNG state). */
typedef struct bflbm_params {
  double kBT;
  double tau_f, tau_g;
  double alpha0, alpha1;
  double kappa;
  double rho_lo, rho_hi;
  unsigned long long seed;
  long long step0;
} bflbm_params;

typedef struct bflbm_lattice bflbm_lattice; /* opaque */

/* shipped defaults: kBT 0, tau 1/2, alpha0 4, alpha1 0, kappa 4, rho in [0,1], seed 12345 */
int bflbm_params_default(bflbm_params* p);

/* Whole periodic box nx*ny*nz on CUDA device `device`.
 * Replaces the MultiFab allocation block main_run_job.cpp:190-212 (fold,fnew,gold,gnew,hydrovs,
 * hydrovsbar,fnoisevs,gnoisevs; nghost=2). */
int bflbm_create(const bflbm_params* p, int nx, int ny, int nz, int device, bflbm_lattice** out);

/* One z-slab [z0, z0+nz_local) of a periodic box nx*ny*nz_global.  Replaces BoxArray::maxSize +
 * DistributionMapping (main_run_job.cpp:140-143) by a 1-D slab decomposition. */
int bflbm_create_slab(const bflbm_params* p, int nx, int ny, int nz_global, int z0, int nz_local, int device,
                      bflbm_lattice** out);
int bflbm_destroy(bflbm_lattice* h);

/* Run-time change of the reference's global parameters (they are plain globals there). */
int bflbm_set_params(bflbm_lattice* h, const bflbm_params* p);
int bflbm_get_params(const bflbm_lattice* h, bflbm_params* p);

/* Use the caller's CUDA stream (a cudaStream_t) for all subsequent work; NULL = the library's own. */
int bflbm_set_stream(bflbm_lattice* h, void* cuda_stream);
/* 0 = one-pass fused step (default); 1 = two-pass step (density kernel + collide/stream kernel, whole-box lattices
 * only; kept as an independent cross-check of the fused path). */
int bflbm_set_algorithm(bflbm_lattice* h, int algo);
/* Height (planes) of the CTA bricks of the fused step; 0 = automatic.  Results are bit-identical for any
 * number of slabs as long as every slab uses the same brick height and it divides nz_local. */
int bflbm_set_tiling(bflbm_lattice* h, int brick_lz);

/* LBM_init_mixture  LBM_binary.H:598-629 */
int bflbm_init_mixture(bflbm_lattice* h);
/* LBM_init_stripe   LBM_binary.H:663-695 (frac = main_run_job.cpp:33 init_frac) */
int bflbm_init_stripe(bflbm_lattice* h, double frac);
/* LBM_init_droplet  LBM_binary.H:698-742 (radius = main_run_job.cpp:110) */
int bflbm_init_droplet(bflbm_lattice* h, double radius);
/* LBM_init (restart) LBM_binary.H:631-661.  f,g: host, (19, nz_local, ny, nx); whole-box lattices only. */
int bflbm_init_from_populations(bflbm_lattice* h, const double* f, const double* g);
/* Same for a slab: arrays carry one extra plane below and above, (19, nz_local+2, ny, nx), holding the
 * periodic neighbours' boundary planes (what FillBoundary would put in the first ghost layer). */
int bflbm_init_from_populations_slab(bflbm_lattice* h, const double* f_ghosted, const double* g_ghosted);

/* USE_REF_STATE (LBM_binary.H:12 -- shipped commented out -- and :92-107): the thermal-noise amplitudes are built from the
 * equilibrium profiles rho_eq, phi_eq, rhot_eq read at the cell shifted by the integer part of (centre of mass of rho now -
 * centre of mass of rho_eq), which the library recomputes on the device after every step (update_com, LBM_binary.H:586-588).
 * The arrays are host arrays of the WHOLE box, (nz_global, ny, nx) each, also for a slab: what main_run_job.cpp:216-221 loads
 * from the equilibrium_* plotfiles of the kBT = 0 run.  Every lattice keeps all of them on its device, because the shift is
 * unbounded: 24 B per cell of the whole box (3.2 GB for 512^3, 25.8 GB on each GPU of an 8 x 512^3 box), counted in
 * bflbm_device_bytes.  NULL pointers switch back to the shipped behaviour (amplitudes from the current densities); a null
 * rho_eq with non-null others, or the reverse, is BFLBM_ERR_ARG.
 *   whole box : switches the lattice to the thread-per-cell two-pass kernels (the results of earlier releases);
 *               bflbm_set_algorithm(h, 0) or a brick height then moves it to the one-pass brick kernel with the same noise,
 *               the centre of mass taken inside every step (also inside replayed CUDA graphs).
 *   slab      : brick kernel.  The centre of mass needs every slab, so a slab takes ONE extra exchange per step, after
 *               bflbm_step_end and before the next bflbm_step_begin (and likewise after an init, a restart's halo refresh or
 *               this call on an initialised slab): bflbm_com_buffer is a device array of bflbm_com_doubles = 4 * nz_global
 *               doubles, one {sum rho, sum rho x, sum rho y, sum rho z} per global plane, in which the slab has written its
 *               own planes and zeros everywhere else.  The caller runs an in-place SUM all-reduce of it over all slabs
 *               (MPI_Allreduce, NCCL, device copies), then bflbm_com_update queues the shift on the lattice's stream.  Each
 *               entry has exactly one non-zero contributor, so every slab gets the same bits whatever order the collective
 *               uses, and the shift is bitwise that of the whole box on the brick kernel.  bflbm_step_begin returns
 *               BFLBM_ERR_STATE while the update is pending; bflbm_step_slab refuses reference-state slabs.
 * At kBT = 0 the steps run the plain kernels but the centre of mass is still kept current (for a later kBT > 0).
 * bflbm_get_reference_com: com_ref[0] of main_run_job.cpp:229-233.  bflbm_get_reference_shift: the current integer shift
 * (synchronises the lattice's stream; test hook). */
int bflbm_set_reference_state(bflbm_lattice* h, const double* rho_eq, const double* phi_eq, const double* rhot_eq);
size_t bflbm_com_doubles(const bflbm_lattice* h);
void* bflbm_com_buffer(bflbm_lattice* h);
int bflbm_com_update(bflbm_lattice* h);
int bflbm_get_reference_shift(const bflbm_lattice* h, int* shift3);
int bflbm_get_reference_com(const bflbm_lattice* h, double* com3);

/* LBM_timestep  LBM_binary.H:544-594, nsteps times.  Asynchronous on the lattice's stream.
 * For a slab lattice use bflbm_step_begin / halo exchange / bflbm_step_end instead. */
int bflbm_step(bflbm_lattice* h, int nsteps);
int bflbm_sync(bflbm_lattice* h);
long long bflbm_step_count(const bflbm_lattice* h);
/* geom.Domain() of the lattice: local valid size, first global plane and global height (z0 = 0, nz_global = nz_local
 * for a whole box).  Any pointer may be NULL. */
int bflbm_get_dims(const bflbm_lattice* h, int* nx, int* ny, int* nz_local, int* z0, int* nz_global);

/* fold/gold after the last step (post-stream populations): what the checkpoint writer reads,
 * main_run_job.cpp:399-409. */
int bflbm_get_populations(bflbm_lattice* h, double* f, double* g);
/* hydrovs, 22 components in VariableNames order (AMReX_FileIO.H:208-261; values LBM_binary.H:216-294). */
int bflbm_get_hydrovars(bflbm_lattice* h, double* out22);
/* hydrovsbar components 0-8: rho, phi, ubar_f xyz, rho+phi, ubar_g xyz (LBM_binary.H:329-339). */
int bflbm_get_hydrovars_bar(bflbm_lattice* h, double* out9);
/* fnoisevs/gnoisevs for the NEXT collision (what WriteOutNoise dumps: Debug.H:380-409). */
int bflbm_get_noise(bflbm_lattice* h, double* fn, double* gn);
/* The 33 standard normals per cell behind bflbm_get_noise, shape (nz_local, ny, nx, 33), in the
 * reference's draw order (LBM_binary.H:115-127).  Test hook: lets the CPU oracle be driven with the
 * GPU's random numbers. */
int bflbm_get_normals(bflbm_lattice* h, double* out33);
/* Same getters into DEVICE memory owned by the caller (full local size, same layout). */
int bflbm_get_hydrovars_device(bflbm_lattice* h, double* dev_out22);
int bflbm_get_hydrovars_bar_device(bflbm_lattice* h, double* dev_out9);
/* Same into a DEVICE array of the whole box, (22, nz_global, ny, nx), which may live on another GPU of this process (a peer
 * copy): how the structure-factor accumulator assembles a slab-decomposed field on one device. */
int bflbm_get_hydrovars_device_into_global(bflbm_lattice* h, double* dev_global22);
int bflbm_get_device(const bflbm_lattice* h); /* CUDA device of the lattice */
int bflbm_get_populations_device(bflbm_lattice* h, double* dev_f, double* dev_g);

/* Host arrays of the WHOLE box, shape (ncomp, nz_global, ny, nx) -- the MultiFab a reference driver holds.  A slab reads /
 * writes only its own planes [z0, z0 + nz_local) (for the restart also the two periodic neighbour planes), so every
 * slab of a box can be pointed at the same arrays (ParallelCopy to / from a single-box MultiFab, AMReX_FileIO.H:18-34).
 * After bflbm_init_from_global_populations a slab that is not in peer mode still needs the halo refresh. */
int bflbm_init_from_global_populations(bflbm_lattice* h, const double* f_global, const double* g_global);
int bflbm_get_populations_into_global(bflbm_lattice* h, double* f_global, double* g_global);
int bflbm_get_hydrovars_into_global(bflbm_lattice* h, double* global22);
int bflbm_get_hydrovars_bar_into_global(bflbm_lattice* h, double* global9);
int bflbm_get_noise_into_global(bflbm_lattice* h, double* fn_global, double* gn_global);

/* ---- asynchronous host transfers: ensembles of restarts and output while stepping ----------------------------------------
 * The reference's two-stage workflow starts every fluctuating run from the checkpoint of the kBT = 0 run
 * (LoadSingleMultiFab + LBM_init, main_run_job.cpp:244-268) and writes a frame every plot_int steps (:372-385).  With the calls above both transfers
 * stand between the steps.  These move them next to the steps, on a copy stream of the lattice:
 *   bflbm_stage_populations : starts the host -> device copy of a checkpoint into a staging area on the device and returns at
 *       once; the lattice may be stepping meanwhile.  ghosted = 0: arrays (19, nz_local, ny, nx), whole box (the arguments of
 *       bflbm_init_from_populations); ghosted = 1: (19, nz_local + 2, ny, nx) (those of bflbm_init_from_populations_slab).
 *       The host arrays must stay untouched until bflbm_stage_wait (or bflbm_init_from_staged + bflbm_sync) has returned;
 *       pinned host memory makes the copy truly asynchronous.  One checkpoint can be staged at a time.
 *   bflbm_init_from_staged  : bflbm_init_from_populations[_slab] of the staged checkpoint, bit for bit, queued on the lattice's
 *       stream behind the copy (no host synchronisation).  Consumes the staged checkpoint; the next one may be staged at once.
 *   bflbm_get_hydrovars_async / _bar_async : the observer runs on the lattice's stream into a device buffer, the device -> host
 *       copy on the copy stream; returns at once, steps queued afterwards overlap the copy.  The host array is complete
 *       after bflbm_download_wait.  One download in flight per lattice (a second call waits for the first on the device).
 * Device memory: the staging area (2 x 19 doubles per cell) and the output buffer (9 or 22 per cell) are allocated on first
 * use and kept; bflbm_release_staging frees them. */
int bflbm_stage_populations(bflbm_lattice* h, const double* f, const double* g, int ghosted);
int bflbm_stage_wait(bflbm_lattice* h);
int bflbm_init_from_staged(bflbm_lattice* h);
int bflbm_get_hydrovars_async(bflbm_lattice* h, double* out22);
int bflbm_get_hydrovars_bar_async(bflbm_lattice* h, double* out9);
int bflbm_download_wait(bflbm_lattice* h);
int bflbm_release_staging(bflbm_lattice* h);

/* update_com  LBM_hydrovs.H:26-60 (centre of mass of rho; local-slab partial sums:
 * sums4 = {mass, sum rho*x, sum rho*y, sum rho*z_global}). */
int bflbm_center_of_mass(bflbm_lattice* h, double* com3, double* sums4);
/* Raw material of the droplet shape diagnostics (fittingDropletCovariance, LBM_hydrovs.H:258-335): local-slab partial sums
 * sums10 = {M, sum rho x, sum rho y, sum rho z_global, sum rho xx, yy, zz, xy, xz, yz} with cell indices as coordinates. */
int bflbm_second_moments(bflbm_lattice* h, double* sums10);
/* Whole box: centre of mass, mass-weighted covariance {xx, yy, zz, xy, xz, yz} of rho about it, and its eigenvalues in
 * ascending order (what fittingDropletCovariance returns per frame; Eigen there, closed form here).  Any output may be NULL. */
int bflbm_droplet_covariance(bflbm_lattice* h, double* com3, double* cov6, double* eig3);
/* The same from the ten sums (host arithmetic): add up bflbm_second_moments of all slabs of a box first. */
int bflbm_covariance_from_moments(const double* sums10, double* com3, double* cov6, double* eig3);
/* Droplet (W, R) fit: fittingDropletParams, LBM_hydrovs.H:160-213 (call site main_run_job.cpp:358-369, behind if_print_radius):
 * rho ~ 1/2 (1 + tanh((R - |r - r0|) / sqrt(2W))) fitted by a damped gradient flow of `nstep` steps; the result is the mean of
 * the last `step_window` steps, restarted with a smaller step (up to 10 times) while their spread exceeds undul_ratio.
 * The reference's defaults: step_window 20, undul_ratio 0.01, nstep 400, W0 = kappa, R0 = radius, eta_W = eta_R = 0.2, dt = 0.02.
 * Coordinates: unit cube.  out3 = {W, R, undulation}; *converged = 0 where the reference would throw.  The two lattice
 * integrals of every flow step are device reductions (bflbm_droplet_fit_terms: local partial sums
 * {sum rho (R - r') sech^2((R - r')/s), sum rho sech^2(..), min rho, max rho}, s = sqrt(2W), r0 in unit-cube coordinates). */
int bflbm_fit_droplet(bflbm_lattice* h, int step_window, double undul_ratio, int nstep, double W0, double R0, double eta_W, double eta_R,
                      double dt, double* out3, int* converged);
int bflbm_droplet_fit_terms(bflbm_lattice* h, double W, double R, const double* r0, double* sums4);
/* JRn_Rn, JWn_Rn, JRn_Wn, JWn_Wn, KWn, KRn of externlib.H:203-244, 342-366 (test hook; host arithmetic only) */
int bflbm_debug_fit_coefficients(double W, double R, double eta_W, double eta_R, double dt, double C0, double* out6);
/* sums of rho and phi over the local cells (Debug.H:35-72 / main_run_job.cpp:224-228) */
int bflbm_total_mass(bflbm_lattice* h, double* mass_rho, double* mass_phi);
/* MultiFabNANCheck  Debug.H:136-149: counts non-finite values in the 22 hydro fields.
 * Returns BFLBM_ERR_NAN if count > 0 (never exits). */
int bflbm_check_nan(bflbm_lattice* h, long long* count);

/* ---- slab halo exchange (replaces the 7 FillBoundary calls per step, LBM_binary.H:130-131,312,353,
 * 553-555, by ONE message per neighbour per step) -------------------------------------------------
 * side 0 = towards lower z, side 1 = towards higher z.  A message is bflbm_halo_doubles() float64s.
 *   bflbm_step_begin : collide+stream of the first and last brick row, then pack both outgoing messages, all on the
 *                      lattice's stream; the interior rows are launched on a second, internal stream and run while
 *   (the caller moves send(side) of rank r to recv(1-side) of the neighbour on the lattice's stream: NCCL send/recv or P2P)
 *   bflbm_step_end   : join the interior rows, unpack both messages, finish the density field; the step counter
 *                      advances.  No other call on the lattice is allowed between _begin and _end.
 * bflbm_halo_refresh_begin/_end do the same exchange without stepping (after an init). */
size_t bflbm_halo_doubles(const bflbm_lattice* h);
void* bflbm_halo_send_buffer(bflbm_lattice* h, int side); /* device pointers, valid for the lattice's life */
void* bflbm_halo_recv_buffer(bflbm_lattice* h, int side);
int bflbm_step_begin(bflbm_lattice* h);
int bflbm_step_end(bflbm_lattice* h);
int bflbm_halo_refresh_begin(bflbm_lattice* h);
int bflbm_halo_refresh_end(bflbm_lattice* h);

/* ---- peer mode: the exchange without the caller (replaces FillBoundary, LBM_binary.H:553-555, by stores over NVLink) -------
 * Every slab lattice owns a "mailbox" in device memory (two receive slots per side + arrival flags).  Once both
 * neighbours' mailboxes are connected, the pack kernel of bflbm_step_begin writes each message straight into the
 * neighbour's mailbox (peer-mapped memory: NVLink / NVSwitch stores) and raises its flag; bflbm_step_end waits for the own
 * flags on the device.  No NCCL, no copy kernel, no host synchronisation in the step loop.
 *   same process, several devices : bflbm_peer_connect(h, side, bflbm_peer_mailbox(neighbour), neighbour's device)
 *   one process per GPU           : exchange the 64-byte handles of bflbm_peer_ipc_handle out of band (torch.distributed,
 *                                   MPI, a file) and call bflbm_peer_connect_ipc
 * side 0 / 1 = the neighbour towards lower / higher z on the periodic ring.  All lattices of a box must make the same
 * sequence of exchanges (steps, halo refreshes): messages carry a sequence number.
 * Several slabs driven by ONE stream or one device must call _begin on all of them before the first _end (a wait would
 * otherwise sit in front of the launch that satisfies it); slabs on different devices may use bflbm_step_slab. */
#define BFLBM_IPC_HANDLE_BYTES 64
size_t bflbm_peer_mailbox_bytes(const bflbm_lattice* h);
void* bflbm_peer_mailbox(bflbm_lattice* h);
int bflbm_peer_ipc_handle(bflbm_lattice* h, void* out64);
int bflbm_peer_connect(bflbm_lattice* h, int side, void* neighbour_mailbox, int neighbour_device);
int bflbm_peer_connect_ipc(bflbm_lattice* h, int side, const void* handle64);
int bflbm_peer_connected(const bflbm_lattice* h);
/* LBM_timestep nsteps times on a connected slab: (bflbm_step_begin, bflbm_step_end) x nsteps, asynchronous */
int bflbm_step_slab(bflbm_lattice* h, int nsteps);
/* bflbm_halo_refresh_begin + _end on a connected slab (after bflbm_init_from_populations_slab) */
int bflbm_halo_refresh(bflbm_lattice* h);
/* synchronises and reports whether a device-side wait for a neighbour's message ever timed out (10 s) */
int bflbm_halo_error(bflbm_lattice* h, int* flag);

/* ---- one box on several GPUs of ONE process (the `ngpus` a reference maintainer passes instead of setting up MPI ranks) -----
 * Replaces BoxArray::maxSize + DistributionMapping + FillBoundary (main_run_job.cpp:140-145, LBM_binary.H:553-555): z-slabs,
 * one per device, ring-connected in peer mode.  Host arrays are those of the WHOLE box, (ncomp, nz, ny, nx).  devices = NULL:
 * devices 0 .. ngpus-1.  brick_lz = 0: automatic; results are bit-identical to the one-GPU run when both use the same
 * brick height and it divides every slab.  ngpus = 1 is a plain whole-box lattice.  Errors: bflbm_multi_last_error(). */
typedef struct bflbm_multi bflbm_multi;
int bflbm_multi_create(const bflbm_params* p, int nx, int ny, int nz, int ngpus, const int* devices, int brick_lz, bflbm_multi** out);
int bflbm_multi_destroy(bflbm_multi* m);
int bflbm_multi_count(const bflbm_multi* m);
bflbm_lattice* bflbm_multi_slab(bflbm_multi* m, int i); /* the i-th slab, e.g. for bflbm_get_dims */
int bflbm_multi_set_params(bflbm_multi* m, const bflbm_params* p);
int bflbm_multi_init_mixture(bflbm_multi* m);
int bflbm_multi_init_stripe(bflbm_multi* m, double frac);
int bflbm_multi_init_droplet(bflbm_multi* m, double radius);
int bflbm_multi_init_from_populations(bflbm_multi* m, const double* f, const double* g);
/* bflbm_set_reference_state on every slab (whole-box arrays).  bflbm_multi_step and the inits then run the centre-of-mass
 * exchange themselves: peer copies (cudaMemcpyPeerAsync) of each slab's planes into the others' buffers behind cross-device
 * events, no host synchronisation.  ngpus = 1: the whole-box call (two-pass kernels). */
int bflbm_multi_set_reference_state(bflbm_multi* m, const double* rho_eq, const double* phi_eq, const double* rhot_eq);
int bflbm_multi_step(bflbm_multi* m, int nsteps);
int bflbm_multi_sync(bflbm_multi* m);
long long bflbm_multi_step_count(const bflbm_multi* m);
int bflbm_multi_get_populations(bflbm_multi* m, double* f, double* g);
int bflbm_multi_get_hydrovars(bflbm_multi* m, double* out22);
int bflbm_multi_get_hydrovars_bar(bflbm_multi* m, double* out9);
int bflbm_multi_get_noise(bflbm_multi* m, double* fn, double* gn);
int bflbm_multi_total_mass(bflbm_multi* m, double* mass_rho, double* mass_phi);
int bflbm_multi_second_moments(bflbm_multi* m, double* sums10);
int bflbm_multi_center_of_mass(bflbm_multi* m, double* com3);
int bflbm_multi_droplet_covariance(bflbm_multi* m, double* com3, double* cov6, double* eig3);
int bflbm_multi_fit_droplet(bflbm_multi* m, int step_window, double undul_ratio, int nstep, double W0, double R0, double eta_W, double eta_R,
                            double dt, double* out3, int* converged);
int bflbm_multi_check_nan(bflbm_multi* m, long long* count); /* also reports a timed-out halo wait */
long long bflbm_multi_kernel_launches(const bflbm_multi* m);
size_t bflbm_multi_device_bytes(const bflbm_multi* m);
const char* bflbm_multi_last_error(void);

/* Per-kernel device timing (CUDA events on the lattice's stream around each launch of a step):
 * ms4 = accumulated milliseconds of {collide+stream kernel, density fold / density pass, halo pack, halo unpack},
 * steps = steps accumulated since profiling was switched on.  Off by default (events serialise nothing but
 * cost a little launch overhead).  on = 1 reads the events back after every step (one host synchronisation per step);
 * on = 2 defers the read-back to bflbm_get_profile (or every 128 steps): nothing but the event records enters a timed
 * region.  While profiling is on, steps are plain launches (no graph replay) and slab steps run on one stream. */
int bflbm_set_profiling(bflbm_lattice* h, int on);
int bflbm_get_profile(bflbm_lattice* h, double ms4[4], long long* steps);

/* bookkeeping for bench.py: kernels launched by this lattice since creation, and device bytes held */
long long bflbm_kernel_launches(const bflbm_lattice* h);
size_t bflbm_device_bytes(const bflbm_lattice* h);

/* Philox4x32-10 block function (test hook for known-answer vectors; runs on the device). */
int bflbm_debug_philox(const unsigned int ctr[4], const unsigned int key[2], unsigned int out[4]);

/* Which compiled variant the last step launched (test hook; recorded on the host where the step kernel is launched, nothing
 * runs on the device).  out[14]:
 *   0  algorithm (0 fused, 1 two-pass)       1  threads per CTA
 *   2  tile x    3  tile y                    (fused: brick tx, ty; two-pass: block.x, block.y)
 *   4  planes per CTA                         (fused: brick height lz; two-pass: 1)
 *   5  6  7  CTAs along x, y, z               (fused: bricks bx, by, bz; two-pass: the grid)
 *   8  FULL (nx, ny multiples of the fused tile: no partial-tile predicates; 0 for two-pass)
 *   9  RATE1 (tau_f = tau_g = 1/2 specialisation)   10  NOISE (kBT > 0)
 *   11 fold source (1: the brick-interior planes are staged from the extended boxes of the step before; 0: every plane from R)
 *   12 schedule (0 whole box, 1 slab on one stream, 2 slab with the interior rows overlapping the exchange)
 *   13 replayed from a CUDA graph
 * BFLBM_ERR_STATE before the first step. */
#define BFLBM_LAST_STEP_FIELDS 14
int bflbm_debug_last_step(const bflbm_lattice* h, int out[14]);

/* Deep statistics of the in-kernel Gaussian generator (test hook): the 33 normals of ncells cells over nsteps steps binned on the
 * device.  hist[nbins + 2]: equal bins over [lo, hi), then underflow, overflow; joint[32 * 32]: the two normals of one Box-Muller
 * pair over [-4, 4)^2; moments4: sums of n, n^2, n^3, n^4.  10^10 normals take about a second. */
int bflbm_debug_normal_statistics(unsigned long long seed, long long ncells, long long step0, int nsteps, int nbins, double lo, double hi,
                                  unsigned long long* hist, unsigned long long* joint, double* moments4);

const char* bflbm_last_error(void);
const char* bflbm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BFLBM_H_ */
