/* bflbm_sf_slab.h -- structure factors of a box split over several processes (one z-slab per rank), without ever assembling
 * the box on one device.  Same semantics as bflbm_sf (bflbm_sf.h): the same pair lists and var_scaling, r2c DFT with 1/sqrt(N)
 * per transform, Hermitian completion, fftshift, k = 0 zeroed on request (AMReX_DFT.H:19-183), sample mean on get.
 *
 * Slab FFT with one all-to-all transpose per variable ("round").  On rank r, which owns the planes [zsplit[r], zsplit[r+1]):
 *   begin(v)  (round 0 first runs the observer, bflbm_get_hydrovars_device, into this rank's 22 fields)
 *             batched 2-D D2Z over (ny, nx) of every local plane of variable v -> [z][ky][kx], kx in [0, nxh), nxh = nx/2 + 1;
 *             pack: the kx columns are split into nranks contiguous ranges (remainder to the low ranks); the columns of rank d
 *             go to one contiguous block of the send buffer, laid out [z][ky][kx - kx0_d].
 *   the caller moves the blocks: one all-to-all with the counts of bflbm_sf_slab_layout (MPI_Alltoallv of CUDA-aware MPI,
 *             grouped NCCL send/recv, torch.distributed.all_to_all_single, or device copies for slabs of one process).  The
 *             blocks arrive in rank order, so the receive buffer is already variable v as [z][ky][kx_local] over the whole z.
 *   end(v)    batched 1-D Z2Z along z over the rank's (ky, kx) columns, read straight from the receive buffer;
 *             on the last round A_k conj(B_k) of every pair is added to the running sums and the sample count goes up.
 * The split is along kx because the Hermitian partner of column kx is column nx - kx at (-ky, -kz): the rank that owns a kx
 * range holds everything its output columns need, so get needs no second exchange.
 *
 * Device memory per cell of this rank's slab (n_local = nx ny nz_local cells, an even split, nv distinct variables, np pairs):
 *   176                     the 22 observed fields
 *   + (nxh / nx) * 16 nv    z-transformed half spectra of the rank's kx columns
 *   + (nxh / nx) * 16 np    running sums (Re, Im) of every pair
 *   + (nxh / nx) * 48       2-D output, send and receive buffers of one variable
 *   + one cuFFT work area shared by both plans (cufftSetAutoAllocation(0) + cufftSetWorkArea).
 * With the reference's 22 pairs (16 distinct variables) at 512^3 that is 505 B per cell before the work area.  bflbm_sf_slab_get
 * allocates 2 x 8 B per output column cell for its duration (the rank's columns of one pair, Re and Im).
 * The lattice's own observer staging (allocated by its first getter call) is not counted.
 *
 * Every call returns 0 or a negative bflbm_status: BFLBM_ERR_ARG for bad partitions, pair indices or rounds outside
 * [0, rounds), BFLBM_ERR_STATE for calls out of order.  Nothing exits. */
#ifndef BFLBM_SF_SLAB_H_
#define BFLBM_SF_SLAB_H_

#include <stddef.h>

#include "bflbm.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bflbm_sf_slab bflbm_sf_slab; /* opaque */

/* lat: this rank's slab (or a whole box with nranks = 1).  zsplit[nranks + 1]: every rank's first plane, zsplit[0] = 0 and
 * zsplit[nranks] = nz.  All ranks create with the same pairs (pairA/pairB/var_scaling as in bflbm_sf_create).
 * BFLBM_ERR_ARG if lat's planes are not [zsplit[rank], zsplit[rank + 1]) or nx/2 + 1 < nranks. */
int bflbm_sf_slab_create(bflbm_lattice* lat, int nranks, int rank, const int* zsplit, int npairs, const int* pairA,
                         const int* pairB, const double* var_scaling, bflbm_sf_slab** out);
int bflbm_sf_slab_destroy(bflbm_sf_slab* s);
/* Queue all work of begin / end / reset / get on this cudaStream_t (NULL = the default stream).  The exchange of a round must
 * be ordered on it too: the next begin overwrites the send buffer. */
int bflbm_sf_slab_set_stream(bflbm_sf_slab* s, void* cuda_stream);
/* Exchanges per accumulate: one per distinct variable. */
int bflbm_sf_slab_rounds(const bflbm_sf_slab* s);
/* Counts and displacements of round `round`'s all-to-all, in doubles, one entry per rank (arrays of nranks).  The send and
 * receive buffers hold exactly sum(send_counts) and sum(recv_counts) doubles. */
int bflbm_sf_slab_layout(const bflbm_sf_slab* s, int round, size_t* send_counts, size_t* send_displs, size_t* recv_counts,
                         size_t* recv_displs);
void* bflbm_sf_slab_send_buffer(bflbm_sf_slab* s); /* device pointers on the lattice's GPU, the same for every round */
void* bflbm_sf_slab_recv_buffer(bflbm_sf_slab* s);
/* Round 0 also runs the observer, which returns once the lattice's stream has drained (the fields are those of the last step).
 * Otherwise asynchronous on the stream. */
int bflbm_sf_slab_begin(bflbm_sf_slab* s, int round);
/* After the round's exchange.  Last round: pairs accumulated, samples + 1. */
int bflbm_sf_slab_end(bflbm_sf_slab* s, int round);
int bflbm_sf_slab_reset(bflbm_sf_slab* s);
long long bflbm_sf_slab_samples(const bflbm_sf_slab* s);
/* The half-spectrum columns [kx0, kx0 + nkx) that `rank` owns. */
int bflbm_sf_slab_kx_range(const bflbm_sf_slab* s, int rank, int* kx0, int* nkx);
/* This rank's columns of what bflbm_sf_get writes: host arrays of the WHOLE box, (npairs, nz, ny, nx), shifted k grid.  Only
 * the x columns this rank owns are written (the shifted images of its kx and of their partners nx - kx); the rest is left
 * untouched, so the ranks' parts combine into the whole.  imag may be NULL.  Waits for the result. */
int bflbm_sf_slab_get(bflbm_sf_slab* s, int zero_avg, double* real, double* imag);

#ifdef __cplusplus
}
#endif
#endif /* BFLBM_SF_SLAB_H_ */
