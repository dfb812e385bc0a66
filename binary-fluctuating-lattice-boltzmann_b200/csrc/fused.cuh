// One-pass fused step: pull-stream + hydro + collide (+noise) + store, AND the (rho, phi) field of the
// NEXT step, in a single sweep over the populations (608 B/cell of population traffic, SURVEY.md 8(d)).
//
// Why: the collision at x needs grad rho, grad phi at x (LBM_binary.H:237-240, 254-255), i.e. post-stream
// densities at the 18 neighbours, which are themselves sums of populations streamed from THEIR neighbours:
// a radius-2 dependency hidden in the reference's step (hard part 1 of SURVEY.md section 7).  A second
// sweep over the populations would cost another 304 B/cell.  Instead each CTA scatter-accumulates the
// post-collision populations it has just produced into next-step densities:
//     rho_{n+1}(y) = sum_i f*_i(y - c_i)
//   - along x with warp shuffles, along y and z through a rolling 3-plane shared-memory accumulator;
//   - contributions that leave the CTA's brick go to the brick's private one-cell shell ("extended box") in E.
// The NEXT step reads the boxes directly (fold-in-staging): a CTA owns a brick of tx*ty columns and sweeps lz planes
// upward; the (rho, phi) neighbourhood needed for the gradients lives in a 4-plane shared-memory ring that is filled two
// planes ahead with cp.async -- the brick's own extended plane is one contiguous copy, the entries that also lie in a
// neighbouring brick's box fetch and add those 1 or 3 contributions in a fixed order.  Only the first / last plane of a
// brick (two brick rows contribute) and the slab faces go through k_fold and R.
// No atomics, no zero-fill pass, no separate density pass, bit-reproducible, and independent of how many GPUs the box
// is cut into (as long as slab boundaries are brick boundaries).
// Inside an iteration all 38 pulls are issued first and (rate-1 kernels) the cell's 33 normals are generated in their
// shadow; the measured reasons for this shape, and what was tried instead, are in profiles/README.md.
#pragma once
#include "kernels.cuh"

// build-time experiment knobs of the general-rate kernels (see profiles/README.md)
#ifndef BFLBM_G_NORMALS_EARLY
#define BFLBM_G_NORMALS_EARLY 0
#endif
#ifndef BFLBM_PARK_F
#define BFLBM_PARK_F 0
#endif
#ifndef BFLBM_PARK_G
#define BFLBM_PARK_G 19
#endif
#ifndef BFLBM_G_MOMENT_SPACE   // 1: species g keeps its 15 non-conserved MOMENTS in shared memory (30 KB instead of 38 KB per CTA)
#define BFLBM_G_MOMENT_SPACE 1
#endif
#ifndef BFLBM_F_MOMENT_SPACE   // 1: species f is relaxed in moment space in place (full forward transform, no f_old kept)
#define BFLBM_F_MOMENT_SPACE 1
#endif
#ifndef BFLBM_GENERAL_SEQ      // 1: general rates load g, park it, then load f (fewer registers in flight)
#define BFLBM_GENERAL_SEQ 1
#endif
#ifndef BFLBM_GENERAL_FMA_NOISE  // 1: the general-rate kernels apply the noise in the fma form of the rate-1 kernels
#define BFLBM_GENERAL_FMA_NOISE 0
#endif
#ifndef BFLBM_Y3_LATE            // 1: general rates make the noise key and the momentum normals after the f loads are consumed
#define BFLBM_Y3_LATE 1
#endif
#ifndef BFLBM_F_NORMALS_EARLY
#define BFLBM_F_NORMALS_EARLY 0
#endif

namespace bflbm {

struct BrickGrid {
  int tx, ty, lz;   // brick = tx*ty threads (256), lz planes
  int bx, by, bz;   // bricks per axis (last one may be partial)
  int ex, ey;       // tx+2, ty+2
  int pl;           // ex*ey     : extended plane, in double2
  long long brick;  // pl*(lz+2) : extended box, in double2
};

inline BrickGrid make_brick_grid(const Geom& G, int lz_request = 0, int nthreads = 256, int max_tx = 32) {
  BrickGrid B;
  int tx = 8;
  while (tx < G.nx && tx < max_tx) tx <<= 1;
  B.tx = tx;
  B.ty = nthreads / tx;  // nthreads = CELLS per CTA plane
  B.bx = (G.nx + B.tx - 1) / B.tx;
  B.by = (G.ny + B.ty - 1) / B.ty;
  int lz = lz_request;
  if (lz <= 0) {
    // Bricks as tall as possible (a brick of height lz costs (lz + ~0.6) planes and (lz + 2) / lz of the shell traffic:
    // lz = 4 is 12 % slower than 32 at equal fill), under two conditions measured in profiles/r2m_tiling_sweep.txt: the
    // kernel is bandwidth bound, so one partial wave of >= 0.8 x (148 SMs x 2 CTAs) already saturates HBM (128^3: 256
    // CTAs of height 32 beat 2048 of height 4 by 6 %), and between one and two waves the tail costs more than the
    // shorter bricks (160^3: 500 CTAs lose to 1000).
    const long long slots = 148 * 2;
    lz = 4;
    for (int c = 32; c > 4; c >>= 1) {
      const long long ctas = (long long)B.bx * B.by * ((G.nzl + c - 1) / c);
      if ((ctas >= (slots * 8) / 10 && ctas <= slots) || ctas >= 2 * slots) { lz = c; break; }
    }
  }
  if (lz > G.nzl) lz = G.nzl;
  if (lz < 2) lz = 2;
  B.lz = lz;
  B.bz = (G.nzl + lz - 1) / lz;
  B.ex = B.tx + 2;
  B.ey = B.ty + 2;
  B.pl = B.ex * B.ey;
  B.brick = (long long)B.pl * (lz + 2);
  return B;
}
inline size_t brick_doubles2(const BrickGrid& B) { return (size_t)B.brick * B.bx * B.by * B.bz; }
constexpr int FIX_SLOTS = 200;  // extra contributions of one extended plane: 2*(ex + ey) + 4*12 - ... <= 192 for ex*ey <= 2*NT
inline size_t fused_smem_bytes(const BrickGrid& B, bool rate1, bool noise) {
  return (size_t)7 * B.pl * sizeof(double2) + (size_t)B.pl * sizeof(int4) + (size_t)FIX_SLOTS * sizeof(double2) +
         (rate1 ? 0 : (size_t)((BFLBM_G_MOMENT_SPACE ? 15 : BFLBM_PARK_G) + BFLBM_PARK_F) * B.tx * B.ty * sizeof(double)) +
         ((BFLBM_TRIG_TABLE && noise) ? (size_t)1024 * sizeof(float2) : 0);
}
// fold-in-staging (the step kernel sums the brick contributions itself) needs every cell to lie in at most
// 2 bricks per axis, i.e. no brick of width 1
inline bool fold_in_staging_ok(const Geom& G, const BrickGrid& B) {
  const int lx = G.nx - (B.bx - 1) * B.tx, ly = G.ny - (B.by - 1) * B.ty;  // width of the last (partial) brick
  return lx >= 2 && ly >= 2 && B.pl <= 2 * B.tx * B.ty && (long long)B.by * B.bx * B.brick < 2147483647ll;
}

// Bricks whose extended box contains the column (gx, gy), in the canonical summation order
// (dy: 0,-1,+1; dx: 0,-1,+1 relative to the brick that owns the column): c[dy][dx] = offset (in double2) of the
// entry inside one brick row of E, or -1.  Used by k_fold and by the step kernel's staging table, so that both
// add the same numbers in the same order.
__device__ __forceinline__ void fold_candidates(const Geom& G, const BrickGrid& B, int gx, int gy, int (&c)[3][3]) {
  int nbx[3], ncx[3], nby[3], ncy[3];
  {
    const int b = gx / B.tx, l = gx - b * B.tx, v = min(B.tx, G.nx - b * B.tx);
    const int bm = (b + B.bx - 1) % B.bx, bp = (b + 1) % B.bx;
    nbx[0] = b; ncx[0] = l + 1;
    nbx[1] = (l == 0) ? bm : -1;     ncx[1] = min(B.tx, G.nx - bm * B.tx) + 1;
    nbx[2] = (l == v - 1) ? bp : -1; ncx[2] = 0;
  }
  {
    const int b = gy / B.ty, l = gy - b * B.ty, v = min(B.ty, G.ny - b * B.ty);
    const int bm = (b + B.by - 1) % B.by, bp = (b + 1) % B.by;
    nby[0] = b; ncy[0] = l + 1;
    nby[1] = (l == 0) ? bm : -1;     ncy[1] = min(B.ty, G.ny - bm * B.ty) + 1;
    nby[2] = (l == v - 1) ? bp : -1; ncy[2] = 0;
  }
#pragma unroll
  for (int dy = 0; dy < 3; ++dy)
#pragma unroll
    for (int dx = 0; dx < 3; ++dx)
      c[dy][dx] = (nby[dy] < 0 || nbx[dx] < 0) ? -1 : (nby[dy] * B.bx + nbx[dx]) * (int)B.brick + ncy[dy] * B.ex + ncx[dx];
}

// x-stage of the density scatter for one species.  p: post-collision populations of this thread's cell.
// t[g]: what arrives in this thread's column for the 9 (cy,cz) groups (own cell + left neighbour's +x movers
// + right neighbour's -x movers).  Lanes on the tile faces receive nothing from outside the tile: their adds are
// predicated off (what leaves through a face is exported separately, see ef/eg in the kernel).
// group index: 0 (0,0)  1 (+1,0)  2 (-1,0)  3 (0,+1)  4 (0,-1)  5 (+1,+1)  6 (-1,-1)  7 (+1,-1)  8 (-1,+1)
__device__ __forceinline__ double scatter_x1(double own, double to_right, double to_left, double has_left, double has_right, int width) {
  const double l = __shfl_up_sync(0xffffffffu, to_right, 1, width);
  const double r = __shfl_down_sync(0xffffffffu, to_left, 1, width);
  // has_* are exactly 1.0 or 0.0: the fma is an exact masked add (same rounding as own + l + r)
  return fma(r, has_right, fma(l, has_left, own));
}
__device__ __forceinline__ void scatter_x(const double (&p)[Q], int tx, int width, double (&t)[9]) {
  const double hl = tx != 0 ? 1. : 0., hr = tx != width - 1 ? 1. : 0.;
  t[0] = scatter_x1(p[0], p[1], p[2], hl, hr, width);
  t[1] = scatter_x1(p[3], p[7], p[10], hl, hr, width);
  t[2] = scatter_x1(p[4], p[9], p[8], hl, hr, width);
  t[3] = scatter_x1(p[5], p[15], p[18], hl, hr, width);
  t[4] = scatter_x1(p[6], p[17], p[16], hl, hr, width);
  t[5] = p[11];
  t[6] = p[12];
  t[7] = p[13];
  t[8] = p[14];
}

// 32-bit byte offsets inside one component + one (warp-uniform) 64-bit base per component: the pull addresses
// cost one integer add per direction instead of a 64-bit multiply-add per load.
__device__ __forceinline__ double ld_off(const double* __restrict__ base, unsigned byte_off) {
  return __ldg(reinterpret_cast<const double*>(reinterpret_cast<const char*>(base) + byte_off));
}
__device__ __forceinline__ void st_off(double* __restrict__ base, unsigned byte_off, double v) {
  *reinterpret_cast<double*>(reinterpret_cast<char*>(base) + byte_off) = v;
}

// asynchronous global->shared copies (SASS LDGSTS): the (rho,phi) plane needed two planes ahead is fetched at the
// top of an iteration and lands while the current plane is collided (no registers, no exposed latency)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Base pointer of every population component, as a kernel parameter: the address of a load/store is then
// (constant-bank 64-bit base) + (per-thread 32-bit offset) = IADD3 + IADD3.X, instead of a 64-bit multiply-add
// by the component stride per access (4 instructions x 76 accesses per cell in the first version).
struct PopBases {
  const double* in[2 * Q];
  double* out[2 * Q];
};
inline PopBases make_pop_bases(const Geom& G, const double* X, double* Xn) {
  PopBases P;
  for (int i = 0; i < 2 * Q; ++i) {
    P.in[i] = X + (long long)i * G.comp;
    P.out[i] = Xn + (long long)i * G.comp;
  }
  return P;
}

// Both kernels use the population-space form of the collision (physics.cuh): only the conserved moments of the incoming
// state go through the forward transform, and the old populations enter as (1 - w) f_old after the inverse transform.
// RATE1: both relaxation rates are exactly 1 (tau_f = tau_g = 1/2, the reference's shipped and only documented
// setting): that term vanishes, nothing is kept.  General rates: f_old stays in registers, g_old is parked in shared memory.

// FULL: nx and ny are multiples of the tile, every thread owns a cell (no activity predicates, no divergence code).
// REF (instantiated with NOISE only): USE_REF_STATE noise -- the amplitudes come from RS.eq (whole-box profiles) at the cell shifted
// by RS.shift, read once per CTA so that graph replays see the shift of the step before.  RS is not touched when !REF.
template <bool NOISE, bool RATE1, bool FULL, int NT, bool REF>
__global__ void __launch_bounds__(NT, 512 / NT)
k_step_fused(const __grid_constant__ Geom G, const __grid_constant__ BrickGrid B, const __grid_constant__ DevParams P, long long step_arg,
             const long long* __restrict__ step_dev, const __grid_constant__ PopBases XB, const double2* __restrict__ R,
             const double2* __restrict__ Ein, double2* __restrict__ E, int bz0, int two_ends, const __grid_constant__ RefState RS) {
  static_assert(NOISE || !REF, "the reference state only changes the noise amplitudes");
  // time step of the noise key: by value, plus (launches replayed from a CUDA graph) a counter in device memory that the
  // last kernel of every replayed chunk advances -- the arguments of a captured launch cannot change between replays
  const long long step = step_arg + ((NOISE && step_dev != nullptr) ? *step_dev : 0ll);
  // brick row of this CTA: rows bz0 .. bz0+gridDim.z-1, or (two_ends) the first and the last row of the slab -- the
  // rows whose results the halo message needs, launched first so that the exchange overlaps the interior rows
  const int bZ = two_ends ? (blockIdx.z == 0 ? 0 : B.bz - 1) : bz0 + (int)blockIdx.z;
  extern __shared__ double2 smem[];
  double2* Rs = smem;             // [4][ey][ex] ring of (rho,phi) planes zl-1, zl, zl+1 and the one in flight (zl+2)
  double2* A = smem + 4 * B.pl;   // [3][ey][ex] rolling accumulators of next-step (rho,phi)
  int4* Tab = reinterpret_cast<int4*>(smem + 7 * B.pl);     // [ey][ex] fold table: 3 extra sources + meta per entry
  double2* Fix = smem + 8 * B.pl;                           // [FIX_SLOTS] landing slots of the extra contributions
  double* So = reinterpret_cast<double*>(Fix + FIX_SLOTS);  // [19][NT] incoming populations of species g (!RATE1)
  // (cos, sin) of the 1024 Box-Muller angles (philox.cuh), behind everything else
  const float2* Trig = nullptr;
  constexpr bool TAB = NOISE && BFLBM_TRIG_TABLE;
  if (TAB) {
    float2* t = reinterpret_cast<float2*>(So + (RATE1 ? 0 : ((BFLBM_G_MOMENT_SPACE ? 15 : BFLBM_PARK_G) + BFLBM_PARK_F) * NT));
    fill_trig_table(t, threadIdx.y * B.tx + threadIdx.x, NT);
    Trig = t;
  }
  // rate-1 kernels make all 33 normals in the load shadow; the general kernels (19 more live doubles) make g's 15 late
  constexpr int PARK_F = BFLBM_PARK_F, PARK_G = BFLBM_PARK_G;
  constexpr bool FMA_NOISE = RATE1 || BFLBM_GENERAL_FMA_NOISE;  // how the noise is applied (philox.cuh)
  constexpr bool G_NORMALS_EARLY = RATE1 || BFLBM_G_NORMALS_EARLY, F_NORMALS_EARLY = RATE1 || BFLBM_F_NORMALS_EARLY;
  __shared__ int nfix;
  const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * B.tx + tx;
  const int x0 = blockIdx.x * B.tx, y0 = blockIdx.y * B.ty, zb = bZ * B.lz;
  const int x = x0 + tx, y = y0 + ty;
  const bool active = FULL || (x < G.nx && y < G.ny);
  const int vz = min(B.lz, G.nzl - zb);
  double2* Eb = E + (((long long)bZ * B.by + blockIdx.y) * B.bx + blockIdx.x) * B.brick;

  // Staging of one (rho,phi) plane zl (-1..nzl) of the tile + ring into ring slot s, two entries per thread.
  //  - planes on a brick face in z (first / last plane of a brick, slab ghost planes) come from R, where k_fold
  //    has already summed every contribution (and the halo exchange has merged the neighbour slab's);
  //  - every other plane is FOLDED HERE from the previous step's extended boxes Ein: the own brick's extended
  //    plane has the layout of the ring slot (one contiguous copy), and the entries that also lie in a neighbouring
  //    brick's extended box (2 columns / rows on each face) fetch those 1 or 3 extra contributions into Fix[] and
  //    add them in k_fold's canonical order.  No separate fold pass over the lattice, no R traffic for these planes.
  // The in-plane source offsets are the same for every plane: computed once.
  constexpr int STG = 2;  // pl = (tx+2)(ty+2) <= 2*NT for every tile shape used (tx in 8..32, tx*ty = NT >= 128)
  int soff[STG];
  if (tid == 0) nfix = 0;
  __shared__ int ref_shift[3];
  if (REF && tid < 3) ref_shift[tid] = RS.shift[tid];
  __syncthreads();
#pragma unroll
  for (int j = 0; j < STG; ++j) {
    const int idx = tid + j * NT;
    const int ey = idx / B.ex, exx = idx - ey * B.ex;
    int gx = (x0 - 1 + exx) % G.nx, gy = (y0 - 1 + ey) % G.ny;
    gx = gx < 0 ? gx + G.nx : gx;
    gy = gy < 0 ? gy + G.ny : gy;
    soff[j] = idx < B.pl ? gy * G.nx + gx : -1;
    if (Ein != nullptr && idx < B.pl) {
      int4 t = make_int4(0, 0, 0, 0);
      // entries beyond the ring of a partial tile are never read
      if (exx <= min(B.tx, G.nx - x0) + 1 && ey <= min(B.ty, G.ny - y0) + 1) {
        int c[3][3];
        fold_candidates(G, B, gx, gy, c);
        const int mine = ((int)blockIdx.y * B.bx + (int)blockIdx.x) * (int)B.brick + idx;
        int ext[3] = {0, 0, 0}, n = 0, pos = 0, seen = 0;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            const int o = c[dy][dx];
            if (o < 0) continue;
            if (o == mine) pos = seen;
            else if (n < 3) ext[n++] = o;
            ++seen;
          }
        if (n > 0) {
          const int slot = atomicAdd(&nfix, n);
          t = make_int4(ext[0], ext[1], ext[2], n | (pos << 4) | (slot << 8));
        }
      }
      Tab[idx] = t;
    }
  }
  const double2* Ein_row = Ein + (long long)bZ * B.by * B.bx * B.brick;                         // this brick row of Ein
  const double2* Ein_own = Ein_row + ((long long)blockIdx.y * B.bx + blockIdx.x) * B.brick;    // this brick
  auto from_R = [&](int zl) { const int l = zl - zb; return Ein == nullptr || l <= 0 || l >= vz - 1; };  // CTA-uniform
  auto stage_plane = [&](int zl, int s) {
    if (from_R(zl)) {
      const double2* Rp = R + (long long)(zl + 1) * G.plane;
#pragma unroll
      for (int j = 0; j < STG; ++j)
        if (soff[j] >= 0) cp_async16(Rs + s * B.pl + tid + j * NT, Rp + soff[j]);
    } else {
      const long long pz = (long long)(zl - zb + 1) * B.pl;  // extended plane of zl in every brick of this row
#pragma unroll
      for (int j = 0; j < STG; ++j) {
        const int idx = tid + j * NT;
        if (idx < B.pl) {
          cp_async16(Rs + s * B.pl + idx, Ein_own + pz + idx);
          const int4 t = Tab[idx];
          const int n = t.w & 15, slot = t.w >> 8;
          if (n > 0) cp_async16(Fix + slot, Ein_row + pz + t.x);
          if (n > 1) {
            cp_async16(Fix + slot + 1, Ein_row + pz + t.y);
            cp_async16(Fix + slot + 2, Ein_row + pz + t.z);
          }
        }
      }
    }
  };
  // after cp_async_wait_all(): add the extra contributions of MY entries (their copies were all issued by me)
  auto fold_plane = [&](int zl, int s) {
    if (from_R(zl)) return;
#pragma unroll
    for (int j = 0; j < STG; ++j) {
      const int idx = tid + j * NT;
      if (idx < B.pl) {
        const int4 t = Tab[idx];
        const int n = t.w & 15, pos = (t.w >> 4) & 15, slot = t.w >> 8;
        if (n > 0) {
          const double2 own = Rs[s * B.pl + idx];
          double2 v;
          if (n == 1) {  // two addends: the order does not matter
            const double2 e0 = Fix[slot];
            v = make_double2(own.x + e0.x, own.y + e0.y);
          } else {       // four addends: own goes to position pos of the canonical order
            const double2 e0 = Fix[slot], e1 = Fix[slot + 1], e2 = Fix[slot + 2];
            const double2 a0 = pos == 0 ? own : e0, a1 = pos == 0 ? e0 : (pos == 1 ? own : e1);
            const double2 a2 = pos <= 1 ? e1 : (pos == 2 ? own : e2), a3 = pos == 3 ? own : e2;
            v = make_double2(((a0.x + a1.x) + a2.x) + a3.x, ((a0.y + a1.y) + a2.y) + a3.y);
          }
          Rs[s * B.pl + idx] = v;
        }
      }
    }
  };
  for (int idx = tid; idx < 3 * B.pl; idx += NT) A[idx] = make_double2(0., 0.);
  __syncthreads();  // Tab is complete
  stage_plane(zb - 1, 0);
  stage_plane(zb, 1);
  cp_async_commit();
  cp_async_wait_all();
  stage_plane(zb + 1, 2);  // the only prologue plane that can need Fix[]
  cp_async_commit();
  cp_async_wait_all();
  fold_plane(zb + 1, 2);
  __syncthreads();

  const int cell = (ty + 1) * B.ex + (tx + 1);  // this thread's cell in an extended plane
  // byte deltas to the periodic x-1 / x+1 and y-1 / y+1 neighbours (loop invariant):
  // dxv[0] = offset of x+1 minus offset of x (used when c_x = -1, source = x+1), dxv[1] = offset of x-1 minus x
  unsigned dxv[2], dyv[2], c_inpl;
  {
    const int xc = min(x, G.nx - 1), yc = min(y, G.ny - 1);
    dxv[0] = (unsigned)((xc == G.nx - 1 ? -(G.nx - 1) : 1) * 8);
    dxv[1] = (unsigned)((xc == 0 ? (G.nx - 1) : -1) * 8);
    dyv[0] = (unsigned)((yc == G.ny - 1 ? -(G.ny - 1) : 1) * G.nx * 8);
    dyv[1] = (unsigned)((yc == 0 ? (G.ny - 1) : -1) * G.nx * 8);
    c_inpl = (unsigned)(yc * G.nx + xc) * 8u;
  }
  const unsigned pl8 = (unsigned)G.plane * 8u;
  for (int k = 0; k < vz; ++k) {
    const int zl = zb + k;
    // ring slot of plane zl + d : (k + 1 + d) & 3 ; accumulator slot of plane zl + d : (k + 1 + d) % 3
    const int r_m = k & 3, r_0 = (k + 1) & 3, r_p = (k + 2) & 3, r_n = (k + 3) & 3;
    const int s_m = k % 3, s_0 = (k + 1) % 3, s_p = (k + 2) % 3;
    // plane zl+2 goes into the slot that held plane zl-2 (free since the barriers of the previous iteration)
    if (zl + 2 <= G.nzl) stage_plane(zl + 2, r_n);
    cp_async_commit();
    double tf[9], tg[9];
    double ef[5], eg[5];  // edge exports (left face on lane 0, right face on lane tx-1)
    const bool left = tx == 0;
    {
      double mf[Q], mg[Q];
      double fo[Q];  // incoming populations of species f: weight (1 - w_f) in the result (general rates only)
      double gk[(BFLBM_G_MOMENT_SPACE ? 0 : Q - PARK_G) + 1];  // ... and the few of species g that do not wait in shared memory
      float ybg[15];
      unsigned c = 0;  // byte offset of this cell inside a component
      CollideCtx C;
      NoiseKey nk;
      if (active) {
        // gradients first (LBM_binary.H:134-150): only 6 doubles stay live across the population loads (moving them into
        // the load shadow as well was measured: +2.5 % without noise)
        double grho[3], gphi[3];
        {
          double nr[Q], np[Q];
          nr[0] = np[0] = 0.;
          const int sl[3] = {r_m, r_0, r_p};
#pragma unroll
          for (int i = 1; i < Q; ++i) {
            const double2 v = Rs[sl[1 + cz(i)] * B.pl + cell + cy(i) * B.ex + cx(i)];
            nr[i] = v.x;
            np[i] = v.y;
          }
          gradient19(nr, grho);
          gradient19(np, gphi);
        }
        // byte offsets of the 19 pull sources (x - c_i) inside a component; < 4 GiB is checked at creation
        unsigned off[Q];
        {
          c = (unsigned)(zl + 1) * pl8 + c_inpl;
          const unsigned dz[3] = {0u - pl8, 0u, pl8};
#pragma unroll
          for (int i = 0; i < Q; ++i) {  // source = cell - c_i ; unsigned arithmetic wraps consistently
            unsigned o = c;
            if (cz(i) != 0) o += dz[1 - cz(i)];
            if (cy(i) != 0) o += dyv[(1 + cy(i)) >> 1];
            if (cx(i) != 0) o += dxv[(1 + cx(i)) >> 1];
            off[i] = o;
          }
        }
        float y3[3], ybf[15];
        double ref3[3];
        {
          double go[Q];
          // all 38 pulls are issued first; the cell's random numbers -- pure arithmetic on its counter -- are generated
          // in their shadow, before the first loaded value is touched
#pragma unroll
          for (int i = 0; i < Q; ++i) go[i] = ld_off(XB.in[Q + i], off[i]);
          if (RATE1 || !BFLBM_GENERAL_SEQ) {
#pragma unroll
            for (int i = 0; i < Q; ++i) fo[i] = ld_off(XB.in[i], off[i]);
          }
          if (REF) {  // the three equilibrium values travel with the pulls
            const long long n = G.plane * G.nz_global, rc = ref_offset(G, ref_shift[0], ref_shift[1], ref_shift[2], x, y, zl);
#pragma unroll
            for (int k = 0; k < 3; ++k) ref3[k] = __ldg(RS.eq + k * n + rc);
          }
          constexpr bool Y3_LATE = !RATE1 && BFLBM_Y3_LATE;
          if (!Y3_LATE) {
            nk = make_noise_key(P.keys, (unsigned long long)cell_global(G, x, y, zl), step);
            momentum_normals<NOISE, TAB>(nk, y3, Trig);
          }
          if (F_NORMALS_EARLY) mode_normals<NOISE, 0, TAB>(nk, ybf, Trig);
          if (G_NORMALS_EARLY) mode_normals<NOISE, 1, TAB>(nk, ybg, Trig);
          // only the conserved moments (density, momentum) of the incoming state are needed (physics.cuh, collide_species):
          // the rest of the forward transform is dead code
          moments(go, mg);
          if (!RATE1) {  // general rates: the incoming state of g waits in shared memory while f is processed
            if (BFLBM_G_MOMENT_SPACE) {
#pragma unroll
              for (int a = 4; a < Q; ++a) So[(a - 4) * NT + tid] = mg[a];
            } else {
#pragma unroll
              for (int i = 0; i < PARK_G; ++i) So[i * NT + tid] = go[i];
#pragma unroll
              for (int i = PARK_G; i < Q; ++i) gk[i - PARK_G] = go[i];
            }
          }
          if (!RATE1 && BFLBM_GENERAL_SEQ) {
#pragma unroll
            for (int i = 0; i < Q; ++i) fo[i] = ld_off(XB.in[i], off[i]);
          }
          moments(fo, mf);
          if (Y3_LATE) {
            nk = make_noise_key(P.keys, (unsigned long long)cell_global(G, x, y, zl), step);
            momentum_normals<NOISE, TAB>(nk, y3, Trig);
          }
          if (!RATE1) {  // ... and so do the first PARK_F incoming populations of f (register pressure at the inverse transform)
#pragma unroll
            for (int i = 0; i < PARK_F; ++i) So[(PARK_G + i) * NT + tid] = fo[i];
          }
        }
        collide_prepare<NOISE, FMA_NOISE>(P, grho, gphi, y3, mf, mg, C, REF ? ref3 : nullptr);
        if (!F_NORMALS_EARLY) mode_normals<NOISE, 0, TAB>(nk, ybf, Trig);
        collide_species<NOISE, 0, RATE1, !RATE1 && BFLBM_F_MOMENT_SPACE, FMA_NOISE>(P, ybf, C, mf);
      } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) mf[i] = fo[i] = 0.;
      }
      double p[Q];
      populations(mf, p);
      if (!RATE1 && !BFLBM_F_MOMENT_SPACE) {
        const double kf = keep_of(P, 0);
#pragma unroll
        for (int i = 0; i < Q; ++i) p[i] = fma(kf, (i < PARK_F && active) ? So[(PARK_G + i) * NT + tid] : fo[i], p[i]);
      }
      if (active) {
#pragma unroll
        for (int i = 0; i < Q; ++i) st_off(XB.out[i], c, p[i]);
      }
      scatter_x(p, tx, B.tx, tf);
      // what leaves through the left face (lane 0) / right face (lane tx-1); unused on the other lanes
      ef[0] = left ? p[2] : p[1]; ef[1] = left ? p[10] : p[7]; ef[2] = left ? p[8] : p[9];
      ef[3] = left ? p[18] : p[15]; ef[4] = left ? p[16] : p[17];
      if (active) {
        if (!RATE1 && BFLBM_G_MOMENT_SPACE) {  // moment space, in place: m <- (1 - w) m_old + v, then one inverse transform
#pragma unroll
          for (int a = 4; a < Q; ++a) mg[a] = So[(a - 4) * NT + tid];
        }
        if (!G_NORMALS_EARLY) mode_normals<NOISE, 1, TAB>(nk, ybg, Trig);
        collide_species<NOISE, 1, RATE1, !RATE1 && BFLBM_G_MOMENT_SPACE, FMA_NOISE>(P, ybg, C, mg);
      } else {
#pragma unroll
        for (int i = 0; i < Q; ++i) mg[i] = 0.;
      }
      populations(mg, p);
      if (!RATE1 && !BFLBM_G_MOMENT_SPACE && active) {
        const double kg = keep_of(P, 1);
#pragma unroll
        for (int i = 0; i < Q; ++i) p[i] = fma(kg, i < PARK_G ? So[i * NT + tid] : gk[i - PARK_G], p[i]);
      }
      if (active) {
#pragma unroll
        for (int i = 0; i < Q; ++i) st_off(XB.out[Q + i], c, p[i]);
      }
      scatter_x(p, tx, B.tx, tg);
      eg[0] = left ? p[2] : p[1]; eg[1] = left ? p[10] : p[7]; eg[2] = left ? p[8] : p[9];
      eg[3] = left ? p[18] : p[15]; eg[4] = left ? p[16] : p[17];
    }
    // a tile narrower than two lanes would need both faces on one lane; tx >= 8 always
    const bool edge = (tx == 0) || (tx == B.tx - 1);
    const int ecell = (ty + 1) * B.ex + (tx == 0 ? 0 : B.tx + 1);

    cp_async_wait_all();  // my part of plane zl+2 has landed; the barriers below publish it to the CTA
    if (zl + 2 <= G.nzl) fold_plane(zl + 2, r_n);
    __syncthreads();      // S0: the write-out of the previous iteration is finished
    auto add = [&](int slot, int at, double a, double b) {
      double2 v = A[slot * B.pl + at];
      v.x += a;
      v.y += b;
      A[slot * B.pl + at] = v;
    };
    // phase cy = 0 : own row.  groups 0 (cz 0), 3 (cz +1), 4 (cz -1)
    add(s_0, cell, tf[0], tg[0]);
    add(s_p, cell, tf[3], tg[3]);
    add(s_m, cell, tf[4], tg[4]);
    if (edge) {
      add(s_0, ecell, ef[0], eg[0]);
      add(s_p, ecell, ef[3], eg[3]);
      add(s_m, ecell, ef[4], eg[4]);
    }
    __syncthreads();
    // phase cy = +1 : row above.  groups 1 (cz 0), 5 (cz +1), 7 (cz -1)
    add(s_0, cell + B.ex, tf[1], tg[1]);
    add(s_p, cell + B.ex, tf[5], tg[5]);
    add(s_m, cell + B.ex, tf[7], tg[7]);
    if (edge) add(s_0, ecell + B.ex, ef[1], eg[1]);
    __syncthreads();
    // phase cy = -1 : row below.  groups 2 (cz 0), 8 (cz +1), 6 (cz -1)
    add(s_0, cell - B.ex, tf[2], tg[2]);
    add(s_p, cell - B.ex, tf[8], tg[8]);
    add(s_m, cell - B.ex, tf[6], tg[6]);
    if (edge) add(s_0, ecell - B.ex, ef[2], eg[2]);
    __syncthreads();
    // plane zl-1 has received everything this brick can give it: write it out (extended plane k) and recycle
    for (int idx = tid; idx < B.pl; idx += NT) {
      Eb[(long long)k * B.pl + idx] = A[s_m * B.pl + idx];
      A[s_m * B.pl + idx] = make_double2(0., 0.);
    }
  }
  __syncthreads();
  // the two planes still in flight: zl = zb+vz-1 (extended plane vz) and the top shell (vz+1)
  for (int idx = tid; idx < B.pl; idx += NT) {
    Eb[(long long)vz * B.pl + idx] = A[(vz % 3) * B.pl + idx];
    Eb[(long long)(vz + 1) * B.pl + idx] = A[((vz + 1) % 3) * B.pl + idx];
  }
}

// (rho,phi)(x,y,zl) = sum over the bricks whose extended box contains the cell, fixed order
// (dz: 0,-1,+1; dy: 0,-1,+1; dx: 0,-1,+1), grouped per dz so that the part a neighbouring slab contributes
// (dz = -1 at the bottom plane, +1 at the top plane) is ONE addend: bit-identical for any slab count.
// zl = -1 and zl = nzl give this slab's contribution to the neighbour's boundary plane.
// Launched brick-wise like the step kernel (grid = bricks, thread = column, loop over the brick's planes): the
// in-plane candidate list of a column is loop invariant, so a plane costs a handful of predicated 16-byte loads and
// no integer division (the first, cell-per-thread version spent ~250 instructions per cell and ran at 2.6 TB/s).
// MODE 0: every plane.  MODE 1: only what the step kernel does not fold itself -- the first and last plane of every
// brick and the two slab-face outputs (zl = -1, nzl).  MODE 2: the complement of MODE 1 (on demand, for the observers).
// MODE 3 + MODE 4 = MODE 1 split for the overlapped slab step: 3 = the four planes at the slab faces (zl = -1, 0,
// nzl-1, nzl: all the halo message needs, computable from the first and last brick row alone; launched with two
// z-blocks), 4 = the remaining brick-face planes.
// MODE 5 = MODE 1 for a WHOLE-BOX lattice, with the periodic self-exchange folded in (the lattice is its own z-neighbour):
// the thread that sums plane 0 also sums this lattice's contribution to "the upper neighbour's" boundary plane and stores
// boundary = local + remote, ghost = remote + local (the operand order of k_merge_density_halo, hence bit-identical to any slab
// decomposition); likewise at the top.  One extra z-layer of CTAs copies the 5+5 population planes that stream across the
// periodic face into the ghost planes, and its first thread advances the device-side step counter (CUDA-graph replays).
// A whole-box step is then TWO launches (k_step_fused, k_fold<5>); it was 10, then 3, in round 1.
template <int MODE>
__global__ void __launch_bounds__(256, 4) k_fold(Geom G, BrickGrid B, const double2* __restrict__ E, double2* __restrict__ R,
                                                  double* X = nullptr, long long* step_dev = nullptr, int step_bump = 0) {
  const int bX = blockIdx.x, bY = blockIdx.y, bZ = MODE == 3 ? (blockIdx.z == 0 ? 0 : B.bz - 1) : (int)blockIdx.z;
  const int lx = threadIdx.x, ly = threadIdx.y;
  const int x = bX * B.tx + lx, y = bY * B.ty + ly;
  if (MODE == 5 && step_dev != nullptr && (blockIdx.x | blockIdx.y) == 0 && blockIdx.z == B.bz && (lx | ly) == 0) *step_dev += step_bump;
  if (x >= G.nx || y >= G.ny) return;
  if (MODE == 5 && bZ == B.bz) {  // ghost planes of the populations that cross the periodic face
    const long long i = (long long)y * G.nx + x, top = (long long)G.nzl * G.plane;
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        double* Xc = X + (long long)(s * Q + q) * G.comp + i;
        if (cz(q) == 1) Xc[0] = Xc[top];                  // pulled from the plane below: ghost plane 0 <- plane nzl-1
        if (cz(q) == -1) Xc[top + G.plane] = Xc[G.plane];  // ghost plane nzl <- plane 0
      }
    return;
  }
  int inpl[3][3];
  fold_candidates(G, B, x, y, inpl);
  const long long zrow = (long long)B.by * B.bx * B.brick;  // E stride between brick rows in z
  // sum over the in-plane candidates of extended plane ez of brick row bz
  auto group = [&](int bz, int ez) {
    const double2* Ez = E + bz * zrow + (long long)ez * B.pl;
    double2 s = __ldg(Ez + inpl[0][0]);  // the own brick always contains the cell
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        if (dy == 0 && dx == 0) continue;
        if (inpl[dy][dx] >= 0) {
          const double2 v = __ldg(Ez + inpl[dy][dx]);
          s.x += v.x;
          s.y += v.y;
        }
      }
    return s;
  };
  const int zb = bZ * B.lz, vz = min(B.lz, G.nzl - zb);
  double2* Rc = R + (long long)y * G.nx + x;
  if (MODE != 2 && MODE != 4 && MODE != 5) {
    // with one brick row, MODE 3 runs a single z-block that owns both faces
    if (bZ == 0 && (MODE != 3 || blockIdx.z == 0)) Rc[0] = group(0, 0);  // zl = -1 : my share of the lower neighbour's boundary plane
    if (bZ == B.bz - 1 && (MODE != 3 || blockIdx.z == gridDim.z - 1)) Rc[(long long)(G.nzl + 1) * G.plane] = group(bZ, vz + 1);  // zl = nzl
  }
  auto plane_value = [&](int l) {
    double2 tot = group(bZ, l + 1);
    if (l == 0 && bZ > 0) {  // a lower brick is always full height
      const double2 s = group(bZ - 1, B.lz + 1);
      tot.x += s.x;
      tot.y += s.y;
    }
    if (l == vz - 1 && bZ + 1 < B.bz) {
      const double2 s = group(bZ + 1, 0);
      tot.x += s.x;
      tot.y += s.y;
    }
    return tot;
  };
  auto plane = [&](int l) { Rc[(long long)(zb + l + 1) * G.plane] = plane_value(l); };
  if (MODE == 5) {
    const bool first = bZ == 0, last = bZ == B.bz - 1;
    const double2 v0 = plane_value(0);
    const double2 v1 = vz > 1 ? plane_value(vz - 1) : v0;
    if (first) {  // r1 + rn1: plane 0 and the ghost plane above the top
      const int vzl = G.nzl - (B.bz - 1) * B.lz;
      const double2 e = group(B.bz - 1, vzl + 1);
      const double2 m = make_double2(v0.x + e.x, v0.y + e.y);
      Rc[G.plane] = m;
      Rc[(long long)(G.nzl + 1) * G.plane] = m;
    } else if (!(last && vz == 1)) {
      Rc[(long long)(zb + 1) * G.plane] = v0;
    }
    if (last) {   // rn + r0: the top plane and the ghost plane below plane 0
      const double2 e = group(0, 0);
      const double2 m = make_double2(v1.x + e.x, v1.y + e.y);
      Rc[(long long)G.nzl * G.plane] = m;
      Rc[0] = m;
    } else if (vz > 1) {
      Rc[(long long)(zb + vz) * G.plane] = v1;
    }
  } else if (MODE == 1) {
    plane(0);
    if (vz > 1) plane(vz - 1);
  } else if (MODE == 3) {  // slab faces: plane 0 of the first row, the last plane of the last row
    if (bZ == 0 && blockIdx.z == 0) plane(0);
    if (bZ == B.bz - 1 && blockIdx.z == gridDim.z - 1 && !(bZ == 0 && vz == 1)) plane(vz - 1);
  } else if (MODE == 4) {  // brick faces that are not slab faces
    if (bZ > 0 && !(bZ == B.bz - 1 && vz == 1)) plane(0);
    if (bZ < B.bz - 1 && vz > 1) plane(vz - 1);
  } else {
    const int lo = MODE == 2 ? 1 : 0, hi = MODE == 2 ? vz - 1 : vz;
#pragma unroll 4
    for (int l = lo; l < hi; ++l) plane(l);
  }
}

// same local sums straight from the populations (after a restart upload, before the first fused step):
// sum_i X_i(x - c_i) over the source planes this slab owns, i = 0..18 in order.
__global__ void __launch_bounds__(256) k_density_partial(Geom G, const double* __restrict__ X, double2* __restrict__ R) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, zl = (int)blockIdx.z - 1;
  if (x >= G.nx || y >= G.ny) return;
  CellIdx I = cell_idx(G, x, y, zl < 0 ? 0 : (zl >= G.nzl ? G.nzl - 1 : zl));
  // rebuild the plane offsets for the true zl (cell_idx clamps nothing; ghost rows are addressable)
  I.zpl[0] = (long long)zl * G.plane;
  I.zpl[1] = (long long)(zl + 1) * G.plane;
  I.zpl[2] = (long long)(zl + 2) * G.plane;
  double rho = 0., phi = 0.;
#pragma unroll
  for (int i = 0; i < Q; ++i) {
    const int zs = zl - cz(i);  // source plane
    if (zs < 0 || zs >= G.nzl) continue;
    const long long a = nbr<-1>(I, i);
    rho += __ldg(X + (long long)i * G.comp + a);
    phi += __ldg(X + (long long)(Q + i) * G.comp + a);
  }
  R[I.zpl[1] + I.yrow[1] + x] = make_double2(rho, phi);
}

// Whole box on one GPU: the lattice is its own z-neighbour, so the halo step (pack x4, unpack x2, merge x2 for a slab) collapses
// into ONE launch with the same arithmetic: ghost planes of the 5+5 populations that stream across the periodic face, and the
// four density planes  R(1) <- R(1) + R(nzl+1),  R(0) <- R(nzl) + R(0),  R(nzl) <- R(nzl) + R(0),  R(nzl+1) <- R(1) + R(nzl+1)
// (boundary = local + remote, ghost = remote + local: the operand order of k_merge_density_halo, hence bit-identical to slabs).
// Matters for small lattices, where a step is launch bound (32^3: 10 launches of ~4 us against 25 us of kernel).
__global__ void __launch_bounds__(256) k_wrap_whole_box(Geom G, double* X, double2* R) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= G.plane) return;
  const long long top = (long long)G.nzl * G.plane;
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      double* Xc = X + (long long)(s * Q + q) * G.comp + i;
      if (cz(q) == 1) Xc[0] = Xc[top];                  // pulled from the plane below: ghost plane 0 <- plane nzl-1
      if (cz(q) == -1) Xc[top + G.plane] = Xc[G.plane];  // ghost plane nzl <- plane 0
    }
  const double2 r0 = R[i], r1 = R[G.plane + i], rn = R[top + i], rn1 = R[top + G.plane + i];
  R[G.plane + i] = make_double2(r1.x + rn1.x, r1.y + rn1.y);
  R[i] = make_double2(rn.x + r0.x, rn.y + r0.y);
  R[top + i] = make_double2(rn.x + r0.x, rn.y + r0.y);
  R[top + G.plane + i] = make_double2(r1.x + rn1.x, r1.y + rn1.y);
}

// ---- halo messages of a slab: ONE pack launch, ONE unpack launch, optionally straight into the neighbour's memory ----------
// message to the neighbour on `side` (0: lower z, 1: upper z), 14 * plane doubles:
//   [10][plane]   the 5+5 populations of my boundary plane that the neighbour pulls across the face
//   [2 * plane]   Pz: my local partial (rho, phi) sums on my boundary plane
//   [2 * plane]   Ez: my contribution to (rho, phi) on the neighbour's boundary plane
// dst[side] is either this lattice's own send buffer (the caller moves it: NCCL / copies) or -- peer mode -- the receive
// slot inside the NEIGHBOUR's mailbox, mapped into this GPU's address space (same process: peer access; other process:
// CUDA IPC): the pack kernel's stores ARE the transfer over NVLink, no copy kernel, no NCCL kernel, nothing to wait for on
// the host.  Arrival is signalled through a sequence number: every thread fences its stores system-wide, the last CTA of
// the grid (atomic counter) then writes `seq` to the neighbour's flag.
struct HaloPack {
  long long pop_src[2][10];        // offsets (doubles) into X of the 10 components' boundary planes, per side
  long long r_bnd[2], r_out[2];    // offsets (doubles) into R of my boundary plane / the plane just outside the slab
  double* dst[2];
  unsigned long long* flag[2];     // peer mode: the neighbour's arrival flag for this message; otherwise null
  unsigned long long seq;
  unsigned int* done;              // CTA counter of this lattice (peer mode)
};
constexpr int HALO_PER_THREAD = 8;  // elements per thread of the pack / unpack kernels (one CTA = 2048 consecutive cells of a plane)
__global__ void __launch_bounds__(256) k_pack_halo(const __grid_constant__ HaloPack H, const double* __restrict__ X,
                                                    const double* __restrict__ R, long long plane) {
  const int j = blockIdx.y, side = blockIdx.z;
  const double* src = j < 10 ? X + H.pop_src[side][j] : (j < 12 ? R + H.r_bnd[side] + (long long)(j - 10) * plane
                                                                    : R + H.r_out[side] + (long long)(j - 12) * plane);
  double* dst = H.dst[side] + (long long)j * plane;
  const long long i0 = (long long)blockIdx.x * (256 * HALO_PER_THREAD) + threadIdx.x;
  double v[HALO_PER_THREAD];
#pragma unroll
  for (int k = 0; k < HALO_PER_THREAD; ++k) v[k] = i0 + k * 256 < plane ? src[i0 + k * 256] : 0.;
#pragma unroll
  for (int k = 0; k < HALO_PER_THREAD; ++k)
    if (i0 + k * 256 < plane) dst[i0 + k * 256] = v[k];
  if (H.flag[0] != nullptr) {
    // the CTA's stores happen before the barrier; thread 0's system-scope fence is cumulative over what it has observed, so the
    // counter increment -- and, from the last CTA, the flags -- become visible to the neighbour GPU only after the data
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      const unsigned total = gridDim.x * gridDim.y * gridDim.z;
      if (atomicAdd(H.done, 1u) == total - 1) {
        *H.done = 0;  // next launch on this stream starts from zero
        __threadfence_system();
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(H.flag[0]), "l"(H.seq) : "memory");
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(H.flag[1]), "l"(H.seq) : "memory");
      }
    }
  }
}

// src[side]: the message that arrived from the neighbour on `side`.  Peer mode: flag[side] is MY arrival flag for it; every CTA
// waits until it shows `seq` (acquire), bounded by a 10 s timeout that sets *err instead of hanging the GPU.
//   j < 10 : ghost plane of one population component      j == 10 : the density merge
//   boundary plane:  R <- local + Ez(neighbour's contribution)      ghost plane:  R <- Pz(neighbour's local) + mine
struct HaloUnpack {
  long long pop_dst[2][10];
  long long r_bnd[2], r_ghost[2];  // offsets in double2 units into R
  const double* src[2];
  const unsigned long long* flag[2];
  unsigned long long seq;
  int* err;
};
__global__ void __launch_bounds__(256) k_unpack_halo(const __grid_constant__ HaloUnpack U, double* __restrict__ X, double2* __restrict__ R,
                                                      long long plane) {
  const long long i0 = (long long)blockIdx.x * (256 * HALO_PER_THREAD) + threadIdx.x;
  const int j = blockIdx.y, side = blockIdx.z;
  if (U.flag[side] != nullptr) {
    if (threadIdx.x == 0) {
      unsigned long long t0 = 0, now, seen;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      for (;;) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(U.flag[side]) : "memory");
        if (seen >= U.seq) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (now - t0 > 10000000000ull) { atomicExch(U.err, 1); break; }
        __nanosleep(200);
      }
    }
    __syncthreads();
  }
  const double* m = U.src[side];
#pragma unroll
  for (int k = 0; k < HALO_PER_THREAD; ++k) {
    const long long i = i0 + k * 256;
    if (i >= plane) break;
    if (j < 10) {
      X[U.pop_dst[side][j] + i] = __ldcg(m + (long long)j * plane + i);
    } else {
      const double2 p = __ldcg(reinterpret_cast<const double2*>(m + 10 * plane) + i);
      const double2 e = __ldcg(reinterpret_cast<const double2*>(m + 12 * plane) + i);
      double2 b = R[U.r_bnd[side] + i], g = R[U.r_ghost[side] + i];
      b.x += e.x; b.y += e.y;
      g.x = p.x + g.x; g.y = p.y + g.y;
      R[U.r_bnd[side] + i] = b;
      R[U.r_ghost[side] + i] = g;
    }
  }
}

// receiving side of the density part of a halo message:
//   boundary plane:  R <- local + Ez(neighbour's contribution)      ghost plane:  R <- Pz(neighbour's local) + mine
__global__ void k_merge_density_halo(long long plane, const double2* __restrict__ Pz, const double2* __restrict__ Ez,
                                     double2* __restrict__ Rb, double2* __restrict__ Rg) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  const double2 p = Pz[i], e = Ez[i];
  double2 b = Rb[i], g = Rg[i];
  b.x += e.x; b.y += e.y;
  g.x = p.x + g.x; g.y = p.y + g.y;
  Rb[i] = b;
  Rg[i] = g;
}

}  // namespace bflbm
