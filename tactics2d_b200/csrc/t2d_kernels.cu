// t2d_kernels.cu - sm_100a kernels and the C ABI (include/t2d_b200.h) of the batched tick.
//
// K1  t2d_step_kernel      fused physics -> pose -> dynamic collision (broadphase + filtered
//                          narrowphase) -> static collision against the map tile in shared
//                          memory (uniform-grid broadphase) -> out-of-bound -> status chain.
//                          (+ t2d_drift_kernel: pre-pass for SingleTrackDrift participants.)
// K2  t2d_reset_kernel     masked re-initialisation from a pool of initial states.
// K3  t2d_physics_kernel   flat batch through one physics model (PhysicsModelBase.step).
// K4  t2d_lidar_kernel     single-line lidar of every scenario's ego (per-edge beam windows).
// K5  t2d_control_kernel   NPC controllers: IDM, cruise / adaptive cruise, pure pursuit.
//     t2d_exchange_allgather_kernel   all-gather of the done masks over NVLink peer memory.
//
// Work decomposition of K1: a scenario (M <= 128 participants) is owned by a group of G lanes of
// one warp, 4 consecutive participants per lane (one float4 per state array per lane: coalesced
// 128-bit loads, 4 independent Euler chains per thread for ILP).  G = pow2 >= ceil(M/4), so a
// warp holds 32/G scenarios and every exchange inside a scenario is warp-synchronous: poses go
// through a per-warp shared-memory tile + __syncwarp, reductions through shuffles.  CTAs are
// persistent (grid = SMs x resident CTAs) and stage the static map tile (segments + broadphase
// grid) into shared memory ONCE with a TMA bulk copy (cp.async.bulk + mbarrier) that overlaps
// the first tile's physics.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/t2d_b200.h"
#include "t2d_math.cuh"
#include "t2d_tile.h"

namespace t2d {

#ifndef T2D_K1_MAX_WARPS
#define T2D_K1_MAX_WARPS 8
#endif
constexpr int MAX_WARPS_PER_CTA = T2D_K1_MAX_WARPS;
constexpr int CTA_THREADS = MAX_WARPS_PER_CTA * 32;   // upper bound; the host picks the warps per CTA (pick_wpc)
constexpr int POSE_PER_WARP = 128;      // 32 lanes x 4 participants per lane (PPL, template parameter of K1: 2 or 4)
constexpr int MAP_SMEM_LIMIT = 120 * 1024;

struct StepArgs {
  float *x, *y, *h, *v, *vx, *vy;
  const uint8_t* type_id;
  int32_t* step_count;
  const float* action;
  const float* ego_action;         // [N][2] action of participant 0 of every scenario (overrides its row of `action`), or nullptr
  uint8_t* flags;
  int16_t* hit_index;
  int16_t* hit_segment;
  uint8_t* scn_status;
  uint8_t* done;
  const unsigned char* map_blob;   // device: the tiles' blobs, one after the other; nullptr when no tile has segments
  const uint32_t* tile_off;        // [n_tiles] byte offset of every tile's blob (map table mode)
  const uint16_t* tile_id;         // [N] the tile of every scenario, or nullptr: every scenario uses tile 0
  MapHeader mh;                    // copy of the blob header (grid geometry, section offsets): constant bank
  const Params* table;             // device
  int map_bytes, map_in_smem;
  int n_types;
  int N, M, G;                     // G = lanes per scenario
  int g_shift, mp_shift, ext, n_tiles, wpc, table_bytes;   // launch-shape constants (see the kernel prologue)
  int off_poseA, off_poseB, off_hit, off_queue, off_posx, off_posy, off_qcount, off_bar;   // shared-memory carve
  int n_steps;
  float dt, dt_rem;
  double dt_d, dt_rem_d, interval_d;   // the same steps in double (dynamics / point mass run in fp64)
  int max_step, cfg_flags;
  int do_physics, has_bounds, vec_ok, needs_vel_in;
  int prefetch;                    // L2 prefetch of tile inputs ahead of their loads (see the kernel prologue)
  float bxmin, bxmax, bymin, bymax;
  float rb_max;                    // largest bounding radius in the type table (broadphase threshold)
  const float* goal_target;        // [N][5] cx, cy, heading, half_len, half_wid of the target area, or nullptr
  float* goal_iou;                 // [N]
  float* goal_last_pose;           // [N][4] x, y, heading, valid
  int32_t* goal_noact_count;       // [N]
  float goal_threshold;
  int goal_noact_max;
  long long* dbg_clock;            // optional [n_tiles][8] phase time stamps (T2D_DEBUG_CLOCK); nullptr in production
  float *wheel_f, *wheel_r;        // [N][M] wheel angular speeds of the SingleTrackDrift participants, or nullptr
};

// ---------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy global -> shared, completion signalled on the mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

// ---------------------------------------------------------------------------- vector access
// N consecutive elements of an [N_scn, M] array as ONE load / store of sizeof(T) * N bytes (<= 16).
template <int BYTES> struct VecOf;
template <> struct VecOf<1> { using T = uint8_t; };
template <> struct VecOf<2> { using T = uint16_t; };
template <> struct VecOf<4> { using T = uint32_t; };
template <> struct VecOf<8> { using T = uint2; };
template <> struct VecOf<16> { using T = uint4; };

template <typename T, int N>
__device__ __forceinline__ void ld_vec(const T* p, T (&o)[N]) {
  using V = typename VecOf<sizeof(T) * N>::T;
  const V v = *reinterpret_cast<const V*>(p);
  memcpy(o, &v, sizeof(V));
}
template <typename T, int N>
__device__ __forceinline__ void st_vec(T* p, const T (&o)[N]) {
  using V = typename VecOf<sizeof(T) * N>::T;
  V v;
  memcpy(&v, o, sizeof(V));
  *reinterpret_cast<V*>(p) = v;
}

// ---------------------------------------------------------------------------- pair narrowphase
// A pose is (x, y, heading, c, s, l, w); w < 0 marks a disc of radius l.
struct Pose {
  float x, y, h, c, s, l, w;
};

__device__ __noinline__ bool pair_exact(const Pose a, const Pose b) {
  const bool ca = a.w < 0.0f, cb = b.w < 0.0f;
  if (!ca && !cb) return obb_obb_f64(a.x, a.y, a.h, a.l, a.w, b.x, b.y, b.h, b.l, b.w);
  if (!ca && cb) return obb_circle_f64(a.x, a.y, a.h, a.l, a.w, b.x, b.y, b.l);
  if (ca && !cb) return obb_circle_f64(b.x, b.y, b.h, b.l, b.w, a.x, a.y, a.l);
  return circle_circle_f64(a.x, a.y, a.l, b.x, b.y, b.l);
}

__device__ __forceinline__ bool pair_hit(const Pose& a, const Pose& b) {
  const bool ca = a.w < 0.0f, cb = b.w < 0.0f;
  int r;
  if (!ca && !cb) r = obb_obb_f32(a.x, a.y, a.c, a.s, a.l, a.w, b.x, b.y, b.c, b.s, b.l, b.w);
  else if (!ca && cb) r = obb_circle_f32(a.x, a.y, a.c, a.s, a.l, a.w, b.x, b.y, b.l);
  else if (ca && !cb) r = obb_circle_f32(b.x, b.y, b.c, b.s, b.l, b.w, a.x, a.y, a.l);
  else r = circle_circle_f32(a.x, a.y, a.l, b.x, b.y, b.l);
  if (r < 0) return pair_exact(a, b);
  return r != 0;
}

__device__ __noinline__ bool seg_exact(const Pose a, const float4 sg) {
  if (a.w < 0.0f) return circle_segment_f64(a.x, a.y, a.l, sg.x, sg.y, sg.z, sg.w);
  return obb_segment_f64(a.x, a.y, a.h, a.l, a.w, sg.x, sg.y, sg.z, sg.w);
}

__device__ __forceinline__ bool seg_hit(const Pose& a, const float4 sg) {
  int r = a.w < 0.0f ? circle_segment_f32(a.x, a.y, a.l, sg.x, sg.y, sg.z, sg.w)
                     : obb_segment_f32(a.x, a.y, a.c, a.s, a.l, a.w, sg.x, sg.y, sg.z, sg.w);
  if (r < 0) return seg_exact(a, sg);
  return r != 0;
}

__device__ __noinline__ bool oob_exact(const Pose a, float xmin, float xmax, float ymin, float ymax) {
  return out_of_bound_f64(a.x, a.y, a.h, a.l, a.w, a.w < 0.0f, xmin, xmax, ymin, ymax);
}

// Every model except the fp32 kinematic fast path (one copy of the fp64 code per kernel).  SingleTrackDrift is NOT
// integrated here: its fp64 tyre model needs far more registers than K1's budget (inlined, or even called, from K1 it
// pushed the whole kernel into spilling and cost the other models 3 - 9 %), so t2d_drift_kernel advances those
// participants in a pre-pass and K1 only builds their pose.
__device__ __noinline__ void other_model_step(OneIO& io, const Params& p, int n_steps, double dt, double dt_rem, double interval) {
  if (p.model() == MODEL_DYNAMICS) {
    dynamics_step(io, p, n_steps, dt);
  } else if (p.model() == MODEL_POINTMASS_NEWTON) {
    pointmass_newton_step(io, p, interval);
  } else if (p.model() == MODEL_POINTMASS_EULER) {
    pointmass_euler_step(io, p, n_steps, dt, dt_rem);
  } else {
    sincos_fast(io.h, &io.sh, &io.ch);
  }
}

// Static broadphase, level 1: the clearance field.  One shared-memory load tells whether the pose's
// bounding circle can reach any segment at all (most participants are nowhere near a wall).
// Split in two so that the global byte load can be issued early and consumed late:
// near_fetch returns the quantised clearance under the participant (0 = treat as near: outside the grid but within
// reach of it; 255 = far), near_decide compares it with the bounding radius.
__device__ __forceinline__ unsigned near_fetch(const float ax, const float ay, const float rbound, const MapHeader& mh, const uint8_t* fine,
                                               unsigned& alt) {
  // branch-free (four of these run side by side per lane): the byte under the participant is fetched from a clamped,
  // always valid address and replaced afterwards when the position lies outside the grid.  The cell indices come
  // from the round-to-nearest magic number (rint(f - 1/2) = floor(f) up to a cell boundary, where either neighbour's
  // clearance is a valid lower bound) instead of float -> int conversions on the XU pipe.
  const float r = rbound * 1.0001f + 1e-3f;
  const float fx = (ax - mh.x0) * mh.inv_cell, fy = (ay - mh.y0) * mh.inv_cell;
  const float gxf = (float)mh.gx, gyf = (float)mh.gy;
  const bool inside = fx >= 0.0f && fy >= 0.0f && fx < gxf && fy < gyf;
  const float kf = (float)mh.fine;
  const int nx = mh.gx * mh.fine, ny = mh.gy * mh.fine;
  const float ux = fmaf(inside ? fx : 0.0f, kf, -0.5f), uy = fmaf(inside ? fy : 0.0f, kf, -0.5f);
  int ix = __float_as_int(ux + RINT_MAGIC) - 0x4B400000, iy = __float_as_int(uy + RINT_MAGIC) - 0x4B400000;
  ix = min(max(ix, 0), nx - 1); iy = min(max(iy, 0), ny - 1);
  const unsigned q = (unsigned)__ldg(fine + (size_t)iy * nx + ix);
  // outside the grid: reachable only within r of its box (NaN position: 255, never near)
  const float ox = fmaxf(fmaxf(-fx, fx - gxf), 0.0f), oy = fmaxf(fmaxf(-fy, fy - gyf), 0.0f);
  const unsigned q_out = fmaxf(ox, oy) * mh.cell <= r ? 0u : 255u;
  // The loaded byte is NOT touched here (its first use would stall the lane on the L2 round trip): it is returned as
  // loaded; `alt` says what to take instead - 0xffffffff: nothing (inside the grid), else the value for outside.
  alt = inside ? 0xffffffffu : q_out;
  return q;
}
__device__ __forceinline__ bool near_decide(unsigned q, unsigned alt, const float rbound) {
  const unsigned v = alt == 0xffffffffu ? q : alt;
  return (float)v * CLEAR_QUANT <= rbound * 1.0001f + 1e-3f;
}

// Own pose of participant `idx` back from the warp's shared-memory tile (the hot loops keep only x, y
// and the bounding radius in registers; the rare exact paths re-read the rest).
// The warp's pose tile is addressed by participant slot (scenario slot x padded participants + participant), but laid
// out lane-minor: slot = lane * PPL + i lives at word i * 32 + lane, so that the lanes' stores of their own PPL
// participants are conflict-free (consecutive lanes, consecutive 16-byte words).  psh = log2(PPL).
__device__ __forceinline__ int pslot(int slot, int psh) { return ((slot & ((1 << psh) - 1)) << 5) | (slot >> psh); }

__device__ __forceinline__ Pose load_pose(const float4* poseA, const float4* poseB, int slot, int psh) {
  const int idx = pslot(slot, psh);
  const float4 a = poseA[idx], b = poseB[idx];
  Pose p;
  p.x = a.x; p.y = a.y; p.h = a.w; p.c = b.x; p.s = b.y; p.l = b.z; p.w = b.w;
  return p;
}

constexpr int QCAP = 192;   // per-warp queue: candidate pairs, then static participants (0..127) + undecided segments (128..191)
constexpr int POS_EXT_PER_WARP = 768;   // circularly extended x / y arrays: (32 / G) x EXT floats per warp, EXT = 1.5 MP + 16 rounded up to 4

// Exact test of one candidate pair (tile indices ti, tj of the same scenario); a hit is recorded for both
// ends as the minimum partner index (scenario-local), which is what "first hit in list order" means.
__device__ __noinline__ void pair_resolve(int ti, int tj, int mp_shift, int psh, const float4* poseA, const float4* poseB, int* hitmin) {
  const Pose a = load_pose(poseA, poseB, ti, psh), b = load_pose(poseA, poseB, tj, psh);
  if (pair_hit(a, b)) {
    const int mask = (1 << mp_shift) - 1;
    atomicMin(&hitmin[pslot(ti, psh)], tj & mask);
    atomicMin(&hitmin[pslot(tj, psh)], ti & mask);
  }
}

// Packed fp32 pair operations of the partner loop (T2D_SCALAR_PAIR: measurement builds fall back to two scalar operations).
#if defined(T2D_SCALAR_PAIR)
__device__ __forceinline__ float2 pk_add(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 pk_fma(float2 a, float2 b, float2 c) { return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
#else
__device__ __forceinline__ float2 pk_add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 pk_fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
#endif

// One word of the partner loop = IPW iterations x PPL own participants x 2 partners.  X / Y: the partner positions of
// the word's iterations (two per float2); nx2 / ny2: the lane's own positions, negated; nthr2: minus the squared
// broadphase reach.  The margin of a pair, d^2 - thr, is <= 0 for a candidate; a NaN position (empty slot) gives a NaN
// margin, which neither the minimum nor the comparison picks up.  FIRST: word 0, where the combinations with partner
// offset <= 0 (the lane's own participants and pairs owned by the other end) are left out at compile time.
template <int PPL, bool FIRST>
__device__ __forceinline__ float pair_word_min(const float2 (&X)[16 / PPL], const float2 (&Y)[16 / PPL], const float2 (&nx2)[PPL],
                                               const float2 (&ny2)[PPL], const float2 (&nthr2)[PPL]) {
  float m = INFINITY;
#pragma unroll
  for (int uu = 0; uu < 16 / PPL; ++uu) {
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      const bool v0 = !FIRST || (2 * uu - i >= 1), v1 = !FIRST || (2 * uu + 1 - i >= 1);
      if (!v0 && !v1) continue;
      const float2 dx = pk_add(X[uu], nx2[i]), dy = pk_add(Y[uu], ny2[i]);
      const float2 d2 = pk_fma(dx, dx, pk_fma(dy, dy, nthr2[i]));
      if (v0 && v1) m = fminf(m, fminf(d2.x, d2.y));
      else if (v0) m = fminf(m, d2.x);
      else m = fminf(m, d2.y);
    }
  }
  return m;
}

// The verdict bits of a word whose minimum margin was <= 0: bit ((uu * PPL + i) * 2 + e), the same margins recomputed.
template <int PPL, bool FIRST>
__device__ __forceinline__ unsigned pair_word_bits(const float2 (&X)[16 / PPL], const float2 (&Y)[16 / PPL], const float2 (&nx2)[PPL],
                                                   const float2 (&ny2)[PPL], const float2 (&nthr2)[PPL]) {
  unsigned bits = 0;
#pragma unroll
  for (int uu = 0; uu < 16 / PPL; ++uu) {
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      const bool v0 = !FIRST || (2 * uu - i >= 1), v1 = !FIRST || (2 * uu + 1 - i >= 1);
      if (!v0 && !v1) continue;
      const float2 dx = pk_add(X[uu], nx2[i]), dy = pk_add(Y[uu], ny2[i]);
      const float2 d2 = pk_fma(dx, dx, pk_fma(dy, dy, nthr2[i]));
      if (v0 && d2.x <= 0.0f) bits |= 1u << ((uu * PPL + i) * 2);
      if (v1 && d2.y <= 0.0f) bits |= 2u << ((uu * PPL + i) * 2);
    }
  }
  return bits;
}

// Broadphase slow path.  `bits` holds the distance-test verdicts of four partner-loop iterations of this lane:
// bit ((uu * PPL + i) * 2 + e) = own participant m0 + i against extended slot m0 + 2 (u_base + uu) + e.  Keep the
// combinations whose partner offset q is 1..Mh (every unordered pair once; q <= 0 are the lane's own participants
// or pairs owned by the other end) and push them on the warp's queue.
template <int PPL>
__device__ __forceinline__ void pair_enqueue_bits(unsigned bits, int u_base, int t0, int tb, int m0, int M, int Mh,
                                                  unsigned* queue, int* qcount) {
  while (bits) {
    const int b = __ffs(bits) - 1;
    bits &= bits - 1;
    const int e = b & 1, i = (b >> 1) & (PPL - 1), uu = (b >> 1) / PPL;   // PPL is a power of two
    const int u = u_base + uu;
    const int q = 2 * u + e - i;
    if (q < 1 || q > Mh) continue;
    int pj = m0 + 2 * u + e;          // < 2.5 M: at most two wraps
    if (pj >= M) pj -= M;
    if (pj >= M) pj -= M;
    const int tj = tb + pj;
    // No function call may appear in this loop: a CALL makes the compiler keep only callee-saved registers
    // live across it and rematerialise everything else in every iteration of the partner loop.  When the
    // queue is full the count keeps growing; the caller then falls back to the exhaustive pass.
    const int slot = atomicAdd(qcount, 1);
    if (slot < QCAP) queue[slot] = ((unsigned)(t0 + i) << 16) | (unsigned)tj;
  }
}

// Dense-scene fallback (the candidate queue overflowed): every lane resolves all pairs of its own participants
// against all partners of the scenario directly.  Correct for any density, slow, and never on the hot path.
template <int PPL>
__device__ __noinline__ void pair_exhaustive(int t0, int tb, int m0, int M, int mp_shift, float rb_max, const float4* poseA,
                                             const float4* poseB, int* hitmin) {
  constexpr int psh = PPL == 4 ? 2 : 1;
  for (int i = 0; i < PPL; ++i) {
    if (m0 + i >= M) break;
    const float4 a = poseA[pslot(t0 + i, psh)];
    if (!(a.x == a.x)) continue;
    const float rr = a.z + rb_max;
    for (int j = m0 + i + 1; j < M; ++j) {
      const float4 b = poseA[pslot(tb + j, psh)];
      const float dx = b.x - a.x, dy = b.y - a.y;
      if (fmaf(dx, dx, dy * dy) <= fmaf(rr * rr, 1.00001f, 1e-12f)) pair_resolve(t0 + i, tb + j, mp_shift, psh, poseA, poseB, hitmin);
    }
  }
}

// Static level 2 for ONE participant (tile index ti), run by one lane: walk the grid cells under the bounding
// circle, fp32-filtered segment test per listed segment, keep the lowest hit.  No function call in here (see
// pair_enqueue_bits): a segment the filter cannot decide is pushed on the exact queue (entries QX0 .. QCAP-1
// of the warp's queue, counter qcount) and decided after the loop; if that queue is full the participant is
// marked (returns -2) for the out-of-line exact walk.
constexpr int QX0 = 128;   // first exact-queue entry (entries below hold the compacted participant list)

// Static level 2 for ONE participant whose reach is <= the map's dilation: ONE cell look-up (the cell under the centre)
// and one loop over its dilated list.  Returns the lowest hit, 0x7fffffff for none, -2 when the participant needs the
// out-of-line walk (reach beyond the dilation, or the exact queue is full).
__device__ __forceinline__ int static_walk(int ti, const Pose& a, float rbound, const MapHeader& mh, const MapView& mv, unsigned* queue,
                                           int* qcount) {
  const float r = rbound * 1.0001f + 1e-3f;
  if (!(r <= mh.dil)) return -2;
  const float fx = (a.x - mh.x0) * mh.inv_cell, fy = (a.y - mh.y0) * mh.inv_cell;
  if (!(fx >= 0.0f && fy >= 0.0f && fx < (float)mh.gx && fy < (float)mh.gy)) return 0x7fffffff;   // beyond the grown box: out of reach
  const int cx = min((int)fx, mh.gx - 1), cy = min((int)fy, mh.gy - 1);
  const int cidx = cy * mh.gx + cx;
  const uint32_t b = mv.dcell_start[cidx], e = mv.dcell_start[cidx + 1];
  int best = 0x7fffffff;
  bool overflow = false;
  // the pose's bounding circle as a box: a listed segment whose own box misses it (most of a dilated list in a dense map)
  // is skipped for 8 instructions instead of running the 35-instruction filtered test to the same "disjoint" verdict
  const float bx0 = a.x - r, bx1 = a.x + r, by0 = a.y - r, by1 = a.y + r;
  for (uint32_t k = b; k < e; ++k) {
    const int sidx = mv.ditems[k];
    const float4 sg = mv.seg[sidx];
    if (fmaxf(sg.x, sg.z) < bx0 || fminf(sg.x, sg.z) > bx1 || fmaxf(sg.y, sg.w) < by0 || fminf(sg.y, sg.w) > by1) continue;
    const int rr = a.w < 0.0f ? circle_segment_f32(a.x, a.y, a.l, sg.x, sg.y, sg.z, sg.w)
                              : obb_segment_f32(a.x, a.y, a.c, a.s, a.l, a.w, sg.x, sg.y, sg.z, sg.w);
    if (rr > 0) {
      best = sidx;   // the list is ascending: the first hit is the lowest
      break;
    } else if (rr < 0) {
      const int slot = atomicAdd(qcount, 1);
      if (slot < QCAP - QX0) queue[QX0 + slot] = ((unsigned)ti << 16) | (unsigned)sidx;
      else overflow = true;
    }
  }
  return overflow ? -2 : best;
}

// Area polygons (StaticCollision.update tests pose.intersects(area.geometry), collision.py:37-43): a pose that touches no
// edge still intersects the closed polygon when it lies inside it.  `best` = the lowest edge hit so far (0x7fffffff: none);
// returns the first segment of the first OBJECT hit: an edge hit is renamed to its object's first segment, and every ring
// that starts below that and contains the pose centre takes over.  The crossing-number test runs in fp32: it is only
// decisive for rings none of whose edges touch the pose, i.e. whose edges all stay at least the pose's inradius away from
// the centre - far beyond fp32 rounding.
__device__ __noinline__ int static_objects(int best, float px, float py, const MapHeader& mh, const unsigned char* blob) {
  if (best != 0x7fffffff && best >= 0) best = reinterpret_cast<const uint16_t*>(blob + mh.off_objfirst)[best];
  const int32_t* pstart = reinterpret_cast<const int32_t*>(blob + mh.off_poly);
  const float4* pbox = reinterpret_cast<const float4*>(blob + mh.off_pbox);
  const float4* seg = reinterpret_cast<const float4*>(blob + mh.off_seg);
  for (int p = 0; p < mh.n_poly; ++p) {
    const int s0 = pstart[p];
    if (s0 >= best) break;
    const float4 bb = pbox[p];
    if (!(px >= bb.x && px <= bb.y && py >= bb.z && py <= bb.w)) continue;
    bool in = false;
    for (int i = s0; i < pstart[p + 1]; ++i) {
      const float4 e = seg[i];
      if ((e.y > py) != (e.w > py) && px < (e.z - e.x) * (py - e.y) / (e.w - e.y) + e.x) in = !in;
    }
    if (in) { best = s0; break; }
  }
  return best;
}

// Out-of-line exact walk for a participant whose undecided segments did not fit the exact queue (never on the
// hot path): the same cells, every test through the fp32 filter + fp64 fallback.
__device__ __noinline__ int static_walk_exact(const Pose a, float rbound, const MapHeader mh, const float4* seg, const uint32_t* cell_start,
                                              const uint16_t* items) {
  const float r = rbound * 1.0001f + 1e-3f;
  int cx0 = max((int)floorf((a.x - r - mh.x0) * mh.inv_cell), 0), cx1 = min((int)floorf((a.x + r - mh.x0) * mh.inv_cell), mh.gx - 1);
  int cy0 = max((int)floorf((a.y - r - mh.y0) * mh.inv_cell), 0), cy1 = min((int)floorf((a.y + r - mh.y0) * mh.inv_cell), mh.gy - 1);
  int best = 0x7fffffff;
  for (int cy = cy0; cy <= cy1; ++cy)
    for (int cx = cx0; cx <= cx1; ++cx) {
      const int cidx = cy * mh.gx + cx;
      for (uint32_t k = cell_start[cidx]; k < cell_start[cidx + 1]; ++k) {
        const int sidx = items[k];
        if (sidx >= best) break;
        if (seg_hit(a, seg[sidx])) best = sidx;
      }
    }
  return best;
}

// The static phase of one warp tile.  (1) every lane decides with the clearance field which of its participants
// can reach a wall at all; (2) those participants are compacted into a list with warp ballots; (3) the list is
// processed one participant per lane (static_walk), so the divergent cell walks of ~15 % of the participants run
// side by side instead of one after the other; (4) the few filter-undecided segments are settled in fp64.
// Where a participant's tile lives: one tile for everybody (header in the kernel's constant bank, sections in shared or
// global memory), or a table of tiles indexed by the participant's scenario (headers and sections in global memory).
struct TileRef {
  const MapHeader* mh;         // header (constant bank, or global)
  const unsigned char* sec;    // where the sections up to the fine field are read from (shared or global)
  const unsigned char* blob;   // the blob in global memory (fine field, polygon data)
};

template <int PPL, bool MAP_TABLE>
__device__ __forceinline__ void static_phase(unsigned near_bits, int t0, int lane, int tile_first_scn, int mp_shift, const StepArgs& A,
                                             const unsigned char* s_map, const float4* poseA, const float4* poseB, int* segmin,
                                             unsigned* queue, int* qcount) {
  int base = 0;
#pragma unroll
  for (int i = 0; i < PPL; ++i) {
    const bool near = (near_bits >> i) & 1u;
    const unsigned m = __ballot_sync(0xffffffffu, near);
    if (near) queue[base + __popc(m & ((1u << lane) - 1u))] = (unsigned)(t0 + i);
    base += __popc(m);
  }
  constexpr int psh = PPL == 4 ? 2 : 1;
  // the tile of participant slot ti (its scenario = the warp tile's first scenario + ti / padded participants)
  auto tile_of = [&](int ti) {
    TileRef t;
    if constexpr (MAP_TABLE) {
      const long long n = (long long)tile_first_scn + (ti >> mp_shift);
      const unsigned char* blob = A.map_blob + A.tile_off[n < A.N ? A.tile_id[n] : 0];
      t.mh = reinterpret_cast<const MapHeader*>(blob); t.sec = blob; t.blob = blob;
    } else {
      t.mh = &A.mh; t.sec = A.map_in_smem ? s_map : A.map_blob; t.blob = A.map_blob;
    }
    return t;
  };
  __syncwarp();
  for (int k = lane; k < base; k += 32) {
    const int ti = (int)queue[k];
    const TileRef t = tile_of(ti);
    const Pose a = load_pose(poseA, poseB, ti, psh);
    const int best = t.mh->n_seg > 0 ? static_walk(ti, a, poseA[pslot(ti, psh)].z, *t.mh, map_view(t.sec, *t.mh), queue, qcount) : 0x7fffffff;
    segmin[pslot(ti, psh)] = best;   // one lane per participant: plain store (-2 = needs the exact walk)
  }
  __syncwarp();
  const int n_x = min(*qcount, QCAP - QX0);
  for (int k = lane; k < n_x; k += 32) {   // undecided (participant, segment) pairs: exact test
    const unsigned e = queue[QX0 + k];
    const int ti = (int)(e >> 16), sidx = (int)(e & 0xffffu);
    int* sm = &segmin[pslot(ti, psh)];
    if (*sm != -2 && sidx < *sm) {
      const TileRef t = tile_of(ti);
      if (seg_exact(load_pose(poseA, poseB, ti, psh), reinterpret_cast<const float4*>(t.sec + t.mh->off_seg)[sidx])) atomicMin(sm, sidx);
    }
  }
  __syncwarp();
  for (int k = lane; k < base; k += 32) {   // the out-of-line walk where needed; then edges -> objects, polygon containment
    const int ti = (int)queue[k];
    int* sm = &segmin[pslot(ti, psh)];
    const TileRef t = tile_of(ti);
    if (*sm == -2) {
      const MapView mv = map_view(t.sec, *t.mh);
      *sm = static_walk_exact(load_pose(poseA, poseB, ti, psh), poseA[pslot(ti, psh)].z, *t.mh, mv.seg, mv.cell_start, mv.items);
    }
    if (t.mh->n_poly > 0) {
      const float4 pa = poseA[pslot(ti, psh)];
      *sm = static_objects(*sm, pa.x, pa.y, *t.mh, t.blob);
    }
  }
  __syncwarp();
}

__device__ __noinline__ bool oob_slow(const float4* poseA, const float4* poseB, int idx, int psh, float xmin, float xmax, float ymin,
                                      float ymax) {
  const Pose a = load_pose(poseA, poseB, idx, psh);
  int r = out_of_bound_f32(a.x, a.y, a.c, a.s, a.l, a.w, a.w < 0.0f, xmin, xmax, ymin, ymax);
  if (r < 0) r = out_of_bound_f64(a.x, a.y, a.h, a.l, a.w, a.w < 0.0f, xmin, xmax, ymin, ymax) ? 1 : 0;
  return r != 0;
}

// Arrival (arrival.py:32-47) and NoAction (no_action.py:32-53) for the ego of scenario n; returns bit0 = arrived,
// bit1 = no action for more than max_step consecutive ticks.  One lane per scenario, fp64, out of line.
__device__ __noinline__ unsigned ego_goal_events(const StepArgs& A, long long n, float ex, float ey, float eh, float el, float ew) {
  unsigned r = 0;
  float* last = A.goal_last_pose + 4 * n;
  if (A.goal_noact_max > 0) {
    int cnt = A.goal_noact_count[n];
    if (last[3] != 0.0f) {                                          // no_action.py:40-50
      const double iou = rect_iou_f64(ex, ey, eh, el, ew, last[0], last[1], last[2], el, ew);
      cnt = iou > 0.999 ? cnt + 1 : 0;
    }
    A.goal_noact_count[n] = cnt;
    if (cnt > A.goal_noact_max) r |= 2u;                            // no_action.py:53
  }
  last[0] = ex; last[1] = ey; last[2] = eh; last[3] = 1.0f;         // no_action.py:39,51
  const float* tg = A.goal_target + 5 * n;
  const double iou = rect_iou_f64(ex, ey, eh, el, ew, tg[0], tg[1], tg[2], tg[3], tg[4]);   // arrival.py:42-44
  A.goal_iou[n] = (float)iou;
  if (iou >= (double)A.goal_threshold) r |= 1u;                     // arrival.py:45
  return r;
}

// L2 prefetch of the lines a lane's PPL participants will load (state, action, type ids).
__device__ __forceinline__ void prefetch_tile_l2(const StepArgs& A, long long i) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(A.x + i));
  asm volatile("prefetch.global.L2 [%0];" ::"l"(A.y + i));
  asm volatile("prefetch.global.L2 [%0];" ::"l"(A.h + i));
  asm volatile("prefetch.global.L2 [%0];" ::"l"(A.v + i));
  if (A.action) asm volatile("prefetch.global.L2 [%0];" ::"l"(A.action + 2 * i));
  asm volatile("prefetch.global.L2 [%0];" ::"l"(A.type_id + i));
  if (A.needs_vel_in) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(A.vx + i));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(A.vy + i));
  }
}

// ---------------------------------------------------------------------------- K1
// KIN_ONLY: every type in the table is SingleTrackKinematics or static - the fp64 models are compiled out
// (their register footprint would otherwise bound the occupancy of the whole kernel).
#if defined(T2D_K1_MAXNREG)   // experiments: an explicit register budget instead of the launch bounds
#define T2D_K1_BOUNDS __maxnreg__(T2D_K1_MAXNREG)
#else
#define T2D_K1_BOUNDS __launch_bounds__(CTA_THREADS, (PPL == 4 ? 2 : 3))
#endif
// MAP_TABLE: every scenario names its own static-geometry tile (t2d_set_map_table); the tiles are then read from global
// memory, header included.  Otherwise one tile serves all scenarios: header in the constant bank, sections staged into
// shared memory once per CTA.
template <int PPL, bool KIN_ONLY, bool MAP_TABLE>
__global__ void T2D_K1_BOUNDS t2d_step_kernel(const __grid_constant__ StepArgs A) {
  extern __shared__ __align__(128) unsigned char smem[];
  // carve: [map blob | 16B aligned] [type table] [pose tiles, hit mins, queues, positions] [mbarrier]; every
  // offset, shift and count that depends only on the launch shape comes precomputed from the host
  // (kernel-parameter constant bank) instead of integer divisions / loops per thread
  const int map_smem_bytes = (!MAP_TABLE && A.map_in_smem) ? A.map_bytes : 0;
  const int table_bytes = A.table_bytes;
  const int wpc = A.wpc;
  unsigned char* s_map = smem;
  Params* s_table = reinterpret_cast<Params*>(smem + map_smem_bytes);
  float4* s_poseA = reinterpret_cast<float4*>(smem + A.off_poseA);
  float4* s_poseB = reinterpret_cast<float4*>(smem + A.off_poseB);
  int* s_hit = reinterpret_cast<int*>(smem + A.off_hit);
  unsigned* s_queue = reinterpret_cast<unsigned*>(smem + A.off_queue);
  float* s_posx = reinterpret_cast<float*>(smem + A.off_posx);
  float* s_posy = reinterpret_cast<float*>(smem + A.off_posy);
  int* s_qcount = reinterpret_cast<int*>(smem + A.off_qcount);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + A.off_bar);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#if defined(T2D_DEBUG_CLOCK)
  const long long t_entry = A.dbg_clock ? clock64() : 0;
#endif
  // Programmatic dependent launch: let the next tick's grid start launching now (its prologue - shared-memory
  // carve, mbarrier, TMA staging of the static table / map - overlaps this grid's tail) ...
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // Stage the type table and the map tile with TMA bulk copies (UBLKCP) on one mbarrier; the wait sits after
  // the first tile's global loads have been issued, so the staging overlaps the cold HBM reads.
  if (tid == 0) {
    mbar_init(s_bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(s_bar, (uint32_t)(table_bytes + map_smem_bytes));
    bulk_g2s(s_table, A.table, (uint32_t)table_bytes, s_bar);
    if (map_smem_bytes > 0) bulk_g2s(s_map, A.map_blob, (uint32_t)map_smem_bytes, s_bar);
  }
  bool staged = false;
  // L2 prefetch of the first tile's state / action lines while the previous grid drains (its CTAs retire over a
  // microsecond or two; ours take their places one by one and would otherwise just sit in griddepcontrol.wait): L2 is the
  // coherence point of the GPU, so a line fetched early can never be stale when it is loaded after the wait.  Measured
  // at 4096 x 64 with cold inputs: 13.7 -> 12.65 us per tick on one GPU.  With a peer-memory done exchange running under
  // the tick (8 GPUs) the same build measured SLOWER than without the prefetch (16.9 vs 14.25 us per step: the burst of
  // prefetches competes with the exchange kernel's peer stores and system-scope fence, and the exchange chain then sets
  // the pace), so the host leaves it off while an exchange object is alive in the process (T2D_PREFETCH=0 / 1 overrides).
  {
    const long long n_ = ((long long)blockIdx.x * wpc + warp) * (32 >> A.g_shift) + (lane >> A.g_shift);
    const int m_ = (lane & (A.G - 1)) * PPL;
    if (A.prefetch && n_ < A.N && m_ < A.M) prefetch_tile_l2(A, n_ * A.M + m_);   // (inside the arrays: a hint, but no stray addresses)
  }
  // ... and wait here, before the first access to the state the previous tick wrote, until that grid has
  // completed and flushed (no-op when the kernel was not launched as a programmatic dependent).
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int G = A.G, M = A.M;
  const int spw = 32 >> A.g_shift;      // scenarios per warp
  const int sub = lane >> A.g_shift;    // scenario slot inside the warp
  const int gl = lane & (G - 1);        // lane inside the group
  const int m0 = gl * PPL;              // first participant of this lane
  const int MP = G * PPL;               // padded participants per scenario
  // warp-level views of the pose tile; t0 = this lane's first slot in it, tb = its scenario's first slot
  float4* poseA = s_poseA + warp * POSE_PER_WARP;
  float4* poseB = s_poseB + warp * POSE_PER_WARP;
  int* hitmin = s_hit + warp * POSE_PER_WARP;
  unsigned* queue = s_queue + warp * QCAP;
  int* qcount = s_qcount + warp;
  const int tb = sub * MP, t0 = tb + m0;
  const int mp_shift = A.mp_shift;   // MP = 1 << mp_shift
  // circularly extended positions of this scenario: slot k holds participant k mod M, so the partner loop reads
  // consecutive slots (two per 64-bit load) without wrap-around logic
  const int EXT = A.ext;   // (3 MP) / 2 + 16 >= (MP - PPL) + 2 * (partner pairs rounded up to whole words)
  float* posx = s_posx + warp * POS_EXT_PER_WARP + sub * EXT;
  float* posy = s_posy + warp * POS_EXT_PER_WARP + sub * EXT;
  const int Mh = M >> 1;                // partner offsets 1..Mh cover every unordered pair

  const int n_tiles = A.n_tiles;
  for (int tile = (int)blockIdx.x * wpc + warp; tile < n_tiles; tile += (int)gridDim.x * wpc) {
    const long long n = (long long)tile * spw + sub;
    const bool scn_ok = n < A.N;
    int nvalid = scn_ok ? min(PPL, M - m0) : 0;
    if (nvalid < 0) nvalid = 0;
    const long long idx0 = n * M + m0;

#if defined(T2D_DEBUG_CLOCK)   // phase time stamps: measurement builds only (profiles/phase_clocks.py)
    // `dep`: a late result of the phase that ends here.  The (never taken) branch on it cannot be resolved before the value
    // has arrived, so the stamp charges a phase with the latency it creates instead of leaking it into the next one.
    #define T2D_STAMP(k, dep) do { if (A.dbg_clock) { if (__float_as_int((float)(dep)) == 0x7fbfffff) asm volatile("trap;"); \
      if (lane == 0) A.dbg_clock[(long long)tile * 10 + (k)] = clock64(); } } while (0)
#else
    #define T2D_STAMP(k, dep) do { } while (0)
#endif
    T2D_STAMP(0, 0.0f);
    // ------------------------------------------------------------------ load
    float sx[PPL], sy[PPL], shd[PPL], sv[PPL], svx[PPL], svy[PPL], a0[PPL], a1[PPL];
    int tidv[PPL];
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      sx[i] = sy[i] = shd[i] = sv[i] = svx[i] = svy[i] = a0[i] = a1[i] = 0.0f;
      tidv[i] = T2D_TYPE_INACTIVE;
    }
    if (nvalid == PPL && A.vec_ok) {
      ld_vec<float, PPL>(A.x + idx0, sx);
      ld_vec<float, PPL>(A.y + idx0, sy);
      ld_vec<float, PPL>(A.h + idx0, shd);
      ld_vec<float, PPL>(A.v + idx0, sv);
      uint8_t tb8[PPL];
      ld_vec<uint8_t, PPL>(A.type_id + idx0, tb8);
#pragma unroll
      for (int i = 0; i < PPL; ++i) tidv[i] = tb8[i];
      if (A.do_physics) {
        float2 act[PPL];
        if constexpr (PPL == 4) {
          float lo[4], hi[4];
          ld_vec<float, 4>(A.action + 2 * idx0, lo);
          ld_vec<float, 4>(A.action + 2 * idx0 + 4, hi);
          act[0] = make_float2(lo[0], lo[1]); act[1] = make_float2(lo[2], lo[3]);
          act[2] = make_float2(hi[0], hi[1]); act[3] = make_float2(hi[2], hi[3]);
        } else {
          float raw[2 * PPL];
          ld_vec<float, 2 * PPL>(A.action + 2 * idx0, raw);
#pragma unroll
          for (int i = 0; i < PPL; ++i) act[i] = make_float2(raw[2 * i], raw[2 * i + 1]);
        }
#pragma unroll
        for (int i = 0; i < PPL; ++i) { a0[i] = act[i].x; a1[i] = act[i].y; }
        if (A.needs_vel_in) {
          ld_vec<float, PPL>(A.vx + idx0, svx);
          ld_vec<float, PPL>(A.vy + idx0, svy);
        }
      }
    } else {
      // ragged / unaligned rows: predicated scalar loads, fully unrolled (a runtime-indexed loop would demote every
      // per-participant array of this kernel to local memory)
#pragma unroll
      for (int i = 0; i < PPL; ++i) {
        if (i < nvalid) {
          sx[i] = A.x[idx0 + i]; sy[i] = A.y[idx0 + i]; shd[i] = A.h[idx0 + i]; sv[i] = A.v[idx0 + i];
          tidv[i] = A.type_id[idx0 + i];
          if (A.do_physics) {
            a0[i] = A.action[2 * (idx0 + i)]; a1[i] = A.action[2 * (idx0 + i) + 1];
            if (A.needs_vel_in) { svx[i] = A.vx[idx0 + i]; svy[i] = A.vy[idx0 + i]; }
          }
        }
      }
    }
    {   // several tiles per warp (persistent CTAs): the next tile's lines start their way to L2 now
      const long long n_next = n + (long long)gridDim.x * wpc * spw;
      if (A.prefetch && n_next < A.N && m0 < M) prefetch_tile_l2(A, n_next * M + m0);
    }
    if (A.ego_action != nullptr && A.do_physics && gl == 0 && scn_ok) {   // the ego's action comes from its own [N, 2] array
      const float2 ea = reinterpret_cast<const float2*>(A.ego_action)[n];
      a0[0] = ea.x; a1[0] = ea.y;
    }
    if (!staged) {   // table + map tile landed? (first tile only)
      mbar_wait(s_bar, 0);
      staged = true;
    }
    // the participant's type row; its third 16-byte group holds the collision shape and the model / shape ids
    constexpr int psh = PPL == 4 ? 2 : 1;
    float ch[PPL], sh[PPL];
    bool active[PPL], kin[PPL];
    const Params* pp[PPL];
    int model[PPL];
    bool lane_all_kin = true, lane_any_kin = false;
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      active[i] = tidv[i] < A.n_types;
      pp[i] = &s_table[active[i] ? tidv[i] : 0];
      model[i] = pp[i]->model_shape & 0xff;
      kin[i] = active[i] && (model[i] == MODEL_KINEMATICS);
      lane_all_kin = lane_all_kin && kin[i];
      lane_any_kin = lane_any_kin || kin[i];
      ch[i] = 1.0f; sh[i] = 0.0f;
    }
    if (A.cfg_flags & T2D_CFG_STEER_FIRST) {
#pragma unroll
      for (int i = 0; i < PPL; ++i)
        if (model[i] <= MODEL_DYNAMICS || model[i] == MODEL_DRIFT) { float t = a0[i]; a0[i] = a1[i]; a1[i] = t; }
    }

    T2D_STAMP(1, sx[0] + sy[PPL - 1] + shd[0] + sv[PPL - 1] + a0[0] + a1[PPL - 1] + (float)tidv[0]);
    // ------------------------------------------------------------------ physics
    if (A.do_physics) {
      // Kinematic participants of the whole warp advance together in the packed 4-chain loop; slots holding another
      // model (or nothing) ride along on a neutral row (zero speed / action, unbounded ranges) and are discarded.
      if (__any_sync(0xffffffffu, lane_any_kin)) {
        const Params* const null_row = &s_table[A.n_types];
        const Params* pk[PPL];
        KinIO<PPL> io;
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          pk[i] = kin[i] ? pp[i] : null_row;
          io.x[i] = kin[i] ? sx[i] : 0.0f; io.y[i] = kin[i] ? sy[i] : 0.0f;
          io.h[i] = kin[i] ? shd[i] : 0.0f; io.v[i] = kin[i] ? sv[i] : 0.0f;
          io.acc[i] = kin[i] ? a0[i] : 0.0f; io.steer[i] = kin[i] ? a1[i] : 0.0f;
        }
        kinematics_step<PPL>(io, pk, A.n_steps, A.dt, A.dt_rem);
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          if (kin[i]) {
            sx[i] = io.x[i]; sy[i] = io.y[i]; shd[i] = io.h[i]; sv[i] = io.v[i];
            svx[i] = io.vx[i]; svy[i] = io.vy[i]; ch[i] = io.ch[i]; sh[i] = io.sh[i];
          }
        }
      }
      if (!lane_all_kin) {
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          if (active[i] && !kin[i]) {
            if constexpr (!KIN_ONLY) {
              OneIO io;
              io.x = sx[i]; io.y = sy[i]; io.h = shd[i]; io.v = sv[i]; io.vx = svx[i]; io.vy = svy[i];
              io.a0 = a0[i]; io.a1 = a1[i];
              io.ch = 1.0f; io.sh = 0.0f;
              other_model_step(io, *pp[i], A.n_steps, A.dt_d, A.dt_rem_d, A.interval_d);
              sx[i] = io.x; sy[i] = io.y; shd[i] = io.h; sv[i] = io.v; svx[i] = io.vx; svy[i] = io.vy;
              ch[i] = io.ch; sh[i] = io.sh;
            } else {
              sincos_fast(shd[i], &sh[i], &ch[i]);   // static participant: the pose only
            }
          }
        }
      }
      // ---------------------------------------------------------------- store state
      bool all_active = true;
#pragma unroll
      for (int i = 0; i < PPL; ++i) all_active = all_active && active[i];
      if (nvalid == PPL && A.vec_ok && all_active) {   // (an inactive slot keeps its state: vx, vy may not even be loaded)
        st_vec<float, PPL>(A.x + idx0, sx);
        st_vec<float, PPL>(A.y + idx0, sy);
        st_vec<float, PPL>(A.h + idx0, shd);
        st_vec<float, PPL>(A.v + idx0, sv);
        st_vec<float, PPL>(A.vx + idx0, svx);
        st_vec<float, PPL>(A.vy + idx0, svy);
      } else {
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          if (i < nvalid && active[i]) {
            A.x[idx0 + i] = sx[i]; A.y[idx0 + i] = sy[i]; A.h[idx0 + i] = shd[i]; A.v[idx0 + i] = sv[i];
            A.vx[idx0 + i] = svx[i]; A.vy[idx0 + i] = svy[i];
          }
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < PPL; ++i) sincos_fast(shd[i], &sh[i], &ch[i]);
    }

    T2D_STAMP(2, sx[0] + sy[PPL - 1] + ch[0] + sh[PPL - 1] + svx[PPL - 1]);
    // ------------------------------------------------------------------ poses -> shared
    // Only (x, y, bounding radius) stay in registers; the full pose lives in the warp's smem tile.
    float px[PPL], py[PPL], rb[PPL];
    unsigned solid_bits = 0;
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      const Vec4 g2 = params_group(pp[i], 2);             // (pose_l, pose_w, rbound, model | shape << 8): one 128-bit load
      const bool sol = active[i] && (__float_as_int(g2.w) >> 8) != SHAPE_NONE;
      solid_bits |= sol ? (1u << i) : 0u;
      rb[i] = g2.z;                                       // bounding radius, rounded up so the broadphase is conservative
      px[i] = sol ? sx[i] : __int_as_float(0x7fc00000);   // NaN: a non-solid slot never passes a distance test
      py[i] = sy[i];
      // (lane-minor layout, see pslot: these stores are conflict-free)
      poseA[i * 32 + lane] = make_float4(px[i], py[i], rb[i], shd[i]);
      poseB[i * 32 + lane] = make_float4(ch[i], sh[i], g2.x, g2.y);
      hitmin[i * 32 + lane] = 0x7fffffff;
    }
    // circularly extended positions: slot k holds participant k mod M, i.e. this lane's PPL participants go to
    // m0 .. m0 + PPL - 1 and to the copies M and 2 M further on that still fit
    if (m0 < M) {
      if (nvalid == PPL && (M & (PPL - 1)) == 0) {   // whole, aligned groups: one vector store per copy
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int k = m0 + c * M;
          if (k < EXT) { st_vec<float, PPL>(posx + k, px); st_vec<float, PPL>(posy + k, py); }
        }
      } else {
#pragma unroll
        for (int i = 0; i < PPL; ++i)
          if (m0 + i < M)
            for (int k = m0 + i; k < EXT; k += M) { posx[k] = px[i]; posy[k] = py[i]; }
      }
    }
    if (lane == 0) *qcount = 0;
    __syncwarp();
    // the step counter of the status section: fetched here - behind the state stores, so it cannot be hoisted to the top
    // of the tile (where ptxas spilled it, stalling the warp on HBM before its state loads were even issued), and with
    // the whole collision phase in front of its first use
    const int cnt_in = (A.do_physics && gl == 0 && scn_ok) ? A.step_count[n] : 0;

    // static broadphase level 1 (clearance field: one byte per participant through L1/L2), issued here so that
    // its global-load latency hides behind the partner loop
    unsigned near_q[PPL], near_alt[PPL];
#pragma unroll
    for (int i = 0; i < PPL; ++i) { near_q[i] = 255u; near_alt[i] = 255u; }   // 255 = far from every segment
    // this lane's tile (all PPL participants of a lane belong to one scenario)
    const MapHeader* lane_mh = &A.mh;
    const unsigned char* lane_blob = A.map_blob;
    if constexpr (MAP_TABLE) {
      lane_blob = A.map_blob + A.tile_off[scn_ok ? A.tile_id[n] : 0];
      lane_mh = reinterpret_cast<const MapHeader*>(lane_blob);
    }
    if (A.map_blob != nullptr && lane_mh->n_seg > 0) {
#pragma unroll
      for (int i = 0; i < PPL; ++i) {
        unsigned alt;
        near_q[i] = near_fetch(px[i], py[i], rb[i], *lane_mh, lane_blob + lane_mh->off_fine, alt);   // (a NaN position reads cell 0 and is "outside": alt = 255)
        near_alt[i] = ((solid_bits >> i) & 1u) ? alt : 255u;
      }
    }

    T2D_STAMP(3, 0.0f);
    // ------------------------------------------------------------------ dynamic collision
    // Every unordered pair once: participant i tests partners (i+1 .. i+M/2) mod M.  A lane walks the
    // partners of its PPL participants together (one 128-bit pose load per partner, PPL distance tests);
    // candidates (rare) go to the out-of-line narrowphase.  A confirmed hit is recorded for both ends:
    // locally for i, by atomicMin in shared memory for the partner.
    int hit[PPL];
    {
      // hot loop: every lane runs it (idle slots hold NaN and never pass); branch-free; two partners per
      // iteration in packed fp32 (FADD2 / FFMA2).  Per pair the margin d^2 - thr is formed by two fused multiply-adds
      // and folded into a running minimum over the 32 tests of a word (one 3-input FMNMX per partner pair); only a
      // word whose minimum is <= 0 (rare) recomputes its verdict bits and goes to the out-of-line enqueue.
      float2 nx2[PPL], ny2[PPL], nthr2[PPL];
#pragma unroll
      for (int i = 0; i < PPL; ++i) {
        const float rr = rb[i] + A.rb_max;
        const float thr = fmaf(rr * rr, 1.00001f, 1e-12f);   // conservative: any partner's bounding radius <= rb_max
        nx2[i] = make_float2(-px[i], -px[i]);
        ny2[i] = make_float2(-py[i], -py[i]);
        nthr2[i] = make_float2(-thr, -thr);
      }
      // partner pairs u = 0 .. U-1 cover offsets -(PPL-1) .. >= Mh; U is rounded up to whole words (the extended
      // arrays are long enough), so the word body has no bounds test and its loads can be issued back to back
      constexpr int IPW = 16 / PPL;                        // iterations per 32-bit word (2 * PPL bits each)
      const int n_words = Mh > 0 ? (((Mh + PPL + 1) >> 1) + IPW - 1) / IPW : 0;
      const float2* bx = reinterpret_cast<const float2*>(posx + m0);
      const float2* by = reinterpret_cast<const float2*>(posy + m0);
      // one word = 2 * IPW consecutive partners: 128-bit loads when the lane's window is 16-byte aligned (PPL = 4)
      auto load_word = [&](int uw, float2 (&X)[IPW], float2 (&Y)[IPW]) {
        if constexpr (PPL == 4) {
#pragma unroll
          for (int q = 0; q < IPW / 2; ++q) {
            const float4 xv = reinterpret_cast<const float4*>(bx)[uw * (IPW / 2) + q];
            const float4 yv = reinterpret_cast<const float4*>(by)[uw * (IPW / 2) + q];
            X[2 * q] = make_float2(xv.x, xv.y); X[2 * q + 1] = make_float2(xv.z, xv.w);
            Y[2 * q] = make_float2(yv.x, yv.y); Y[2 * q + 1] = make_float2(yv.z, yv.w);
          }
        } else {
#pragma unroll
          for (int uu = 0; uu < IPW; ++uu) { X[uu] = bx[uw * IPW + uu]; Y[uu] = by[uw * IPW + uu]; }
        }
      };
      if (n_words > 0) {   // word 0 also meets the lane's own participants (offset <= 0): those tests are compiled out
        float2 X[IPW], Y[IPW];
        load_word(0, X, Y);
        if (pair_word_min<PPL, true>(X, Y, nx2, ny2, nthr2) <= 0.0f) {
          const unsigned bits = pair_word_bits<PPL, true>(X, Y, nx2, ny2, nthr2);
          if (bits) pair_enqueue_bits<PPL>(bits, 0, t0, tb, m0, M, Mh, queue, qcount);
        }
      }
      for (int uw = 1; uw < n_words; ++uw) {
        float2 X[IPW], Y[IPW];
        load_word(uw, X, Y);
        if (pair_word_min<PPL, false>(X, Y, nx2, ny2, nthr2) <= 0.0f) {
          const unsigned bits = pair_word_bits<PPL, false>(X, Y, nx2, ny2, nthr2);
          if (bits) pair_enqueue_bits<PPL>(bits, uw * IPW, t0, tb, m0, M, Mh, queue, qcount);
        }
      }
      __syncwarp();
      T2D_STAMP(4, *qcount);
      // narrowphase: the queued candidate pairs, one per lane (or the exhaustive pass if the queue overflowed)
      const int n_q = *qcount;
      if (n_q <= QCAP) {
        for (int k = lane; k < n_q; k += 32) {
          const unsigned e = queue[k];
          pair_resolve((int)(e >> 16), (int)(e & 0xffffu), mp_shift, psh, poseA, poseB, hitmin);
        }
      } else {
        pair_exhaustive<PPL>(t0, tb, m0, M, mp_shift, A.rb_max, poseA, poseB, hitmin);
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < PPL; ++i) {
        const int h = hitmin[i * 32 + lane];
        hit[i] = (h == 0x7fffffff) ? -1 : h;
        hitmin[i * 32 + lane] = 0x7fffffff;   // reused below as the per-participant first-hit segment
      }
      if (lane == 0) *qcount = 0;
      __syncwarp();
    }

    T2D_STAMP(5, hit[0] + hit[PPL - 1]);
    // ------------------------------------------------------------------ static collision
    int hseg[PPL];
#pragma unroll
    for (int i = 0; i < PPL; ++i) hseg[i] = -1;
    if (A.map_blob != nullptr) {
      unsigned near_bits = 0;
#pragma unroll
      for (int i = 0; i < PPL; ++i)
        if (((solid_bits >> i) & 1u) && near_decide(near_q[i], near_alt[i], rb[i])) near_bits |= 1u << i;
      if (__any_sync(0xffffffffu, near_bits != 0)) {
        static_phase<PPL, MAP_TABLE>(near_bits, t0, lane, tile * spw, mp_shift, A, s_map, poseA, poseB, hitmin, queue, qcount);
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
          const int h = hitmin[i * 32 + lane];
          hseg[i] = (h == 0x7fffffff) ? -1 : h;
        }
      }
    }

    T2D_STAMP(6, hseg[0] + hseg[PPL - 1]);
    // ------------------------------------------------------------------ out of bound + flags
    // the boundary box of this lane's scenario (Map.boundary of its tile)
    float bxmin = A.bxmin, bxmax = A.bxmax, bymin = A.bymin, bymax = A.bymax;
    bool has_bounds = A.has_bounds != 0;
    if constexpr (MAP_TABLE) {
      has_bounds = lane_mh->has_bounds != 0;
      bxmin = lane_mh->bxmin; bxmax = lane_mh->bxmax; bymin = lane_mh->bymin; bymax = lane_mh->bymax;
    }
    uint8_t fl[PPL];
    unsigned oob_check = 0;   // participants whose bounding circle is not well inside the box (rare): settled below, once
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      uint8_t f = 0;
      if (hit[i] >= 0) f |= T2D_F_DYNAMIC;
      if (hseg[i] >= 0) f |= T2D_F_STATIC;
      // the bounding circle well inside the box: inside for sure (the common case)
      const float r = rb[i] * 1.0001f + 1e-3f;
      const bool clear_in = (px[i] - bxmin > r) && (bxmax - px[i] > r) && (py[i] - bymin > r) && (bymax - py[i] > r);
      if (has_bounds && ((solid_bits >> i) & 1u) && !clear_in) oob_check |= 1u << i;
      fl[i] = f;
    }
    if (oob_check) {
#pragma unroll
      for (int i = 0; i < PPL; ++i)
        if (((oob_check >> i) & 1u) && oob_slow(poseA, poseB, t0 + i, psh, bxmin, bxmax, bymin, bymax)) fl[i] |= T2D_F_OUTBOUND;
    }
    if (nvalid == PPL && A.vec_ok) {
      int16_t h16[PPL], s16[PPL];
#pragma unroll
      for (int i = 0; i < PPL; ++i) { h16[i] = (int16_t)hit[i]; s16[i] = (int16_t)hseg[i]; }
      if (A.flags) st_vec<uint8_t, PPL>(A.flags + idx0, fl);
      if (A.hit_index) st_vec<int16_t, PPL>(A.hit_index + idx0, h16);
      if (A.hit_segment) st_vec<int16_t, PPL>(A.hit_segment + idx0, s16);
    } else {
#pragma unroll
      for (int i = 0; i < PPL; ++i) {
        if (i < nvalid) {
          if (A.flags) A.flags[idx0 + i] = fl[i];
          if (A.hit_index) A.hit_index[idx0 + i] = (int16_t)hit[i];
          if (A.hit_segment) A.hit_segment[idx0 + i] = (int16_t)hseg[i];
        }
      }
    }

    // ------------------------------------------------------------------ scenario status
    if (A.do_physics) {
      unsigned agg;
      if (A.cfg_flags & T2D_CFG_ANY_PARTICIPANT) {
        agg = 0;
#pragma unroll
        for (int i = 0; i < PPL; ++i) agg |= fl[i];
        for (int o = G >> 1; o > 0; o >>= 1) agg |= __shfl_xor_sync(0xffffffffu, agg, o);
      } else {
        agg = __shfl_sync(0xffffffffu, (unsigned)fl[0], sub * G);   // participant 0 = the ego
      }
      if (gl == 0 && scn_ok) {
        const int cnt = cnt_in + 1;                                  // parking.py:353 (loaded with the state)
        A.step_count[n] = cnt;
        uint8_t st = T2D_STATUS_NORMAL;
        unsigned goal = 0;
        if (A.goal_target != nullptr) {   // the ego is participant 0 = this lane's first slot
          const float4 ea = poseA[pslot(t0, psh)], eb = poseB[pslot(t0, psh)];
          if (ea.x == ea.x && eb.w >= 0.0f) goal = ego_goal_events(A, n, ea.x, ea.y, ea.w, eb.z, eb.w);
        }
        if (goal & 1u) st = T2D_STATUS_COMPLETED;                    // parking.py:387-390 (lowest priority)
        if (agg & T2D_F_DYNAMIC) st = T2D_STATUS_FAILED;
        if (agg & T2D_F_STATIC) st = T2D_STATUS_FAILED;              // parking.py:381-385
        if (agg & T2D_F_OUTBOUND) st = T2D_STATUS_OUT_BOUND;         // parking.py:376-379
        if (goal & 2u) st = T2D_STATUS_NO_ACTION;                    // parking.py:371-374
        if (A.max_step > 0 && cnt > A.max_step) st = T2D_STATUS_TIME_EXCEEDED;  // parking.py:366-369
        if (A.scn_status) A.scn_status[n] = st;
        if (A.done) A.done[n] = st != T2D_STATUS_NORMAL;             // parking.py:243-248
      }
    }
    T2D_STAMP(7, fl[0] + fl[PPL - 1]);
#if defined(T2D_DEBUG_CLOCK)
    if (A.dbg_clock && lane == 0) {
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      A.dbg_clock[(long long)tile * 10 + 8] = smid;
      A.dbg_clock[(long long)tile * 10 + 9] = t_entry;
    }
#endif
    __syncwarp();   // pose tile is reused by the next tile
  }
  if (!staged) mbar_wait(s_bar, 0);   // never leave a bulk copy in flight at exit
}

// ---------------------------------------------------------------------------- K2
struct ResetArgs {
  float *x, *y, *h, *v, *vx, *vy;
  int32_t* step_count;
  const uint8_t* mask;
  const int32_t* pool_index;
  const float *px, *py, *ph, *pv, *pvx, *pvy;
  float* goal_last_pose;
  int32_t* goal_noact_count;
  // per-participant state owned by the world besides x .. vy: the SingleTrackDrift wheel speeds and the controllers'
  // State.accel of the previous tick - a new episode must not inherit them from the old one
  float *wheel_f, *wheel_r;            // [N][M] or nullptr
  const float *pool_wf, *pool_wr;      // [n_pool][M] initial wheel speeds, or nullptr: free rolling, speed / wheel radius
  float* last_accel;                   // [N][M] or nullptr
  const uint8_t* type_id;
  const Params* table;
  int n_types;
  int N, M, n_pool;
};

__global__ void t2d_reset_kernel(const __grid_constant__ ResetArgs A) {
  const long long total = (long long)A.N * A.M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / A.M), m = (int)(i - (long long)n * A.M);
    if (!A.mask[n]) continue;
    int r = A.pool_index ? A.pool_index[n] : n;
    r = min(max(r, 0), A.n_pool - 1);
    const long long s = (long long)r * A.M + m;
    A.x[i] = A.px[s]; A.y[i] = A.py[s]; A.h[i] = A.ph[s]; A.v[i] = A.pv[s];
    A.vx[i] = A.pvx ? A.pvx[s] : A.pv[s] * cosf(A.ph[s]);
    A.vy[i] = A.pvy ? A.pvy[s] : A.pv[s] * sinf(A.ph[s]);
    if (A.wheel_f != nullptr) {
      float wf = 0.0f, wr = 0.0f;
      if (A.pool_wf != nullptr) {
        wf = A.pool_wf[s]; wr = A.pool_wr[s];
      } else {
        const int tid = A.type_id[i];
        if (tid < A.n_types && A.table[tid].model() == MODEL_DRIFT) wf = wr = A.pv[s] / A.table[tid].wheel_radius;   // zero slip
      }
      A.wheel_f[i] = wf; A.wheel_r[i] = wr;
    }
    if (A.last_accel != nullptr) A.last_accel[i] = 0.0f;   // a fresh State has no acceleration (state.py:171-185)
    if (m == 0) {
      A.step_count[n] = 0;
      if (A.goal_last_pose) A.goal_last_pose[4 * (long long)n + 3] = 0.0f;   // NoAction.reset / last_pose = None
      if (A.goal_noact_count) A.goal_noact_count[n] = 0;
    }
  }
}

// ---------------------------------------------------------------------------- env epilogue
// What ParkingEnv.step does after check_status (envs/parking.py:240-256, _get_reward :148-190), for all N scenarios in
// one launch: TrafficStatus per participant from the event byte (status.py:52-61), terminated / truncated
// (parking.py:243-248), the reward chain in the reference's order, the two running extrema it keeps per episode
// (_max_iou, _min_dist_to_target) and the done mask that drives the masked reset.  One thread per participant slot;
// the thread of slot 0 also does the per-scenario part.  Reads the ego's flags through the same array, so the launch
// has no other input than the tick's outputs.
struct EnvArgs {
  const uint8_t* flags;        // [N][M] event byte of the tick
  const uint8_t* status;       // [N] ScenarioStatus of the tick
  const int32_t* step_count;   // [N]
  const float *x, *y;          // [N][M] state after the tick (the ego's position for the distance shaping)
  const float* iou;            // [N] IoU(ego pose, target) of the tick, or nullptr (no goal)
  const float* target;         // [N][5] or nullptr
  float* max_iou;              // [N] in/out, or nullptr
  float* min_dist;             // [N] in/out, or nullptr
  float* reward;               // [N]
  uint8_t *terminated, *truncated, *done;   // [N]
  uint8_t* traffic_status;     // [N][M]
  int N, M, max_step, reset_trackers;
};

__global__ void __launch_bounds__(256) t2d_env_epilogue_kernel(const __grid_constant__ EnvArgs A) {
  const long long total = (long long)A.N * A.M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const unsigned f = A.flags[i];
    const uint8_t ts = (f & T2D_F_STATIC) ? 3 : ((f & T2D_F_DYNAMIC) ? 4 : 1);   // COLLISION_STATIC / COLLISION_DYNAMIC / NORMAL
    if (A.traffic_status) A.traffic_status[i] = ts;
    const int n = (int)(i / A.M);
    if (i - (long long)n * A.M != 0) continue;
    const int st = A.status[n];
    // check_status returns at the first detector that fires (parking.py:366-385): the ego's traffic status is only set
    // by the collision detector, i.e. when the scenario status says FAILED
    const int ego_ts = st == T2D_STATUS_FAILED ? ts : 1;
    const bool term = st == T2D_STATUS_COMPLETED;                                  // :243-244
    const bool trunc = !term && (st != T2D_STATUS_NORMAL || ego_ts != 1);          // :245-248
    float r;
    if (ego_ts == 3 || ego_ts == 4) r = -5.0f;                                     // :151-152 (+ dynamic collision, an extension)
    else if (st == T2D_STATUS_TIME_EXCEEDED || st == T2D_STATUS_NO_ACTION) r = -1.0f;   // :153-157
    else if (st == T2D_STATUS_OUT_BOUND) r = -5.0f;                                // :158-159
    else if (st == T2D_STATUS_COMPLETED) r = 5.0f;                                 // :160-161
    else {
      r = A.max_step > 0 ? -tanhf((float)A.step_count[n] / (float)A.max_step) * 0.001f : 0.0f;   // :163
      if (A.iou != nullptr && A.max_iou != nullptr) {
        const float iou = A.iou[n], best = A.max_iou[n];
        r += (best == -INFINITY) ? iou : iou - best;                               // :164-169
        A.max_iou[n] = fmaxf(best, iou);                                           // :170
      }
      if (A.target != nullptr && A.min_dist != nullptr) {
        const float dx = A.x[i] - A.target[5 * (long long)n], dy = A.y[i] - A.target[5 * (long long)n + 1];
        const float d = sqrtf(dx * dx + dy * dy), best = A.min_dist[n];            // :172-185
        if (d < best) {                                                            // :186-188 (inf on the first step: the
          if (best != INFINITY) r += (best - d) * 0.1f;                            //  reference adds inf there; we add nothing)
          A.min_dist[n] = d;
        }
      }
    }
    A.reward[n] = r;
    if (A.terminated) A.terminated[n] = term;
    if (A.truncated) A.truncated[n] = trunc;
    if (A.done) A.done[n] = term || trunc;
    if (A.reset_trackers && (term || trunc)) {   // the next episode starts fresh (ParkingEnv.reset, parking.py:276-277)
      if (A.max_iou) A.max_iou[n] = -INFINITY;
      if (A.min_dist) A.min_dist[n] = INFINITY;
    }
  }
}

// ---------------------------------------------------------------------------- K3
// ---------------------------------------------------------------------------- drift pre-pass
// SingleTrackDrift participants of a tick, one per thread, before K1 (which then only builds their pose).
__global__ void __launch_bounds__(128) t2d_drift_kernel(const __grid_constant__ StepArgs A) {
  const long long total = (long long)A.N * A.M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int tid = A.type_id[i];
    if (tid >= A.n_types) continue;
    const Params& p = A.table[tid];
    if (p.model() != MODEL_DRIFT) continue;
    OneIO io;
    io.x = A.x[i]; io.y = A.y[i]; io.h = A.h[i]; io.v = A.v[i]; io.vx = 0.0f; io.vy = 0.0f;
    float2 act = reinterpret_cast<const float2*>(A.action)[i];
    if (A.ego_action != nullptr && i % A.M == 0) act = reinterpret_cast<const float2*>(A.ego_action)[i / A.M];
    const bool sf = (A.cfg_flags & T2D_CFG_STEER_FIRST) != 0;
    io.a0 = sf ? act.y : act.x; io.a1 = sf ? act.x : act.y;
    io.ch = 1.0f; io.sh = 0.0f;
    io.w0 = A.wheel_f[i]; io.w1 = A.wheel_r[i];
    drift_step(io, p, A.n_steps, A.dt_d, A.dt_rem_d);
    A.x[i] = io.x; A.y[i] = io.y; A.h[i] = io.h; A.v[i] = io.v; A.vx[i] = io.vx; A.vy[i] = io.vy;
    A.wheel_f[i] = io.w0; A.wheel_r[i] = io.w1;
  }
}

struct PhysArgs {
  Params p;
  float *x, *y, *h, *v, *vx, *vy;
  float *wheel_f, *wheel_r;
  const float* action;
  float* applied;
  int n, n_steps;
  float dt, dt_rem;
  double dt_d, dt_rem_d, interval_d;
};

__global__ void __launch_bounds__(256) t2d_physics_kernel(const __grid_constant__ PhysArgs A) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (long long)gridDim.x * blockDim.x) {
    if (A.p.model() == MODEL_KINEMATICS) {
      KinIO<1> io;
      io.x[0] = A.x[i]; io.y[0] = A.y[i]; io.h[0] = A.h[i]; io.v[0] = A.v[i];
      io.acc[0] = A.action[2 * i]; io.steer[0] = A.action[2 * i + 1];
      const Params* const p1[1] = {&A.p};
      kinematics_step<1>(io, p1, A.n_steps, A.dt, A.dt_rem);
      A.x[i] = io.x[0]; A.y[i] = io.y[0]; A.h[i] = io.h[0]; A.v[i] = io.v[0]; A.vx[i] = io.vx[0]; A.vy[i] = io.vy[0];
      if (A.applied) { A.applied[2 * i] = io.acc[0]; A.applied[2 * i + 1] = io.steer[0]; }
    } else {
      OneIO io;
      io.x = A.x[i]; io.y = A.y[i]; io.h = A.h[i]; io.v = A.v[i]; io.vx = A.vx[i]; io.vy = A.vy[i];
      io.a0 = A.action[2 * i]; io.a1 = A.action[2 * i + 1];
      io.ch = 1.0f; io.sh = 0.0f;
      if (A.p.model() == MODEL_DRIFT) {
        io.w0 = A.wheel_f[i]; io.w1 = A.wheel_r[i];
        drift_step(io, A.p, A.n_steps, A.dt_d, A.dt_rem_d);
        A.wheel_f[i] = io.w0; A.wheel_r[i] = io.w1;
      } else {
        other_model_step(io, A.p, A.n_steps, A.dt_d, A.dt_rem_d, A.interval_d);
      }
      A.x[i] = io.x; A.y[i] = io.y; A.h[i] = io.h; A.v[i] = io.v; A.vx[i] = io.vx; A.vy[i] = io.vy;
      if (A.applied) { A.applied[2 * i] = io.a0; A.applied[2 * i + 1] = io.a1; }
    }
  }
}

// ---------------------------------------------------------------------------- K4
// Single-line lidar of the ego (participant 0) of every scenario: SingleLineLidar._scan_obstacles
// (tactics2d/sensor/lidar.py:128-221).  Obstacle edges = the map's collidable segments (the reference takes the
// exteriors of `area.type_ == "obstacle"`, :137-143) + the pose rings of the other box-shaped participants (:146-153;
// a Pedestrian's pose is not a ring and is skipped there too), transformed into the ego frame (:105-126); per beam
// the reference's determinant intersection with its 1e-8 slack box filters (:160-213), min over edges, clip to the
// range, range -> inf.  One warp per scenario: sources are culled by distance, the surviving edges go to shared memory
// together with their beam window (beam_window below), and the warp walks the edges with its lanes sharing the beams of
// each window.  fp64 throughout (from the fp32 state): every tested pair gives exactly the float64 oracle's value, the
// untested pairs are ones the reference's own filters reject.
constexpr int LIDAR_EDGES = 144;   // edges per shared-memory chunk per warp (4 doubles + a beam window each)
constexpr int LIDAR_WARPS = 4;
constexpr int LIDAR_BEAMS = 512;   // beams per pass (running minima in shared memory)

struct LidarArgs {
  const float *x, *y, *h;
  const uint8_t* type_id;
  const Params* table;
  int n_types;
  const unsigned char* map_blob;
  const uint32_t* tile_off;   // map table: byte offsets of the tiles; the scenario's tile id, or nullptr = tile 0 for all
  const uint16_t* tile_id;
  const double* beam_cs;   // [n_beams][2] cos, sin of the beam angles (host float64)
  float* scan;             // [N][n_beams]
  int N, M, n_beams;
  double range;
};

__device__ __forceinline__ double point_segment_dist2(double x1, double y1, double x2, double y2) {   // from the origin
  const double dx = x2 - x1, dy = y2 - y1, dd = dx * dx + dy * dy;
  double t = dd > 0.0 ? -(x1 * dx + y1 * dy) / dd : 0.0;
  t = fmin(fmax(t, 0.0), 1.0);
  const double ex = x1 + t * dx, ey = y1 + t * dy;
  return ex * ex + ey * ey;
}

// (beam_window, the per-edge beam interval, lives in t2d_math.cuh so that tests/hostsim can check it on the host.)
__global__ void __launch_bounds__(LIDAR_WARPS * 32, 7) t2d_lidar_kernel(const __grid_constant__ LidarArgs A) {
  __shared__ double s_edge[LIDAR_WARPS][LIDAR_EDGES][4];
  __shared__ BeamWindow s_win[LIDAR_WARPS][LIDAR_EDGES];
  __shared__ float s_best[LIDAR_WARPS][LIDAR_BEAMS];
  __shared__ int s_cnt[LIDAR_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n = (long long)blockIdx.x * LIDAR_WARPS + warp;
  if (n >= A.N) return;
  double(*edge)[4] = s_edge[warp];
  BeamWindow* win = s_win[warp];
  float* best = s_best[warp];
  int* cnt = &s_cnt[warp];
  const long long base = n * A.M;
  const int t_ego = A.type_id[base];
  float* out = A.scan + n * A.n_beams;
  if (t_ego >= A.n_types) {   // no ego: nothing is seen
    for (int b = lane; b < A.n_beams; b += 32) out[b] = INFINITY;
    return;
  }
  const double x0 = A.x[base], y0 = A.y[base], th = A.h[base];
  double sa, ca;
  sincos(th, &sa, &ca);
  const double xoff = -x0 * ca - y0 * sa, yoff = x0 * sa - y0 * ca;   // lidar.py:116-121
  const double R = A.range, R2 = R * R;
  // the scenario's static-geometry tile (its header is read from global memory: one warp, a handful of words)
  const unsigned char* blob = A.map_blob ? A.map_blob + (A.tile_id ? A.tile_off[A.tile_id[n]] : 0u) : nullptr;
  const MapHeader* tmh = reinterpret_cast<const MapHeader*>(blob);
  const int n_seg = blob ? tmh->n_seg : 0;
  const float4* seg = n_seg > 0 ? reinterpret_cast<const float4*>(blob + tmh->off_seg) : nullptr;
  const int part_rounds = (A.M - 1 + 31) / 32, seg_rounds = (n_seg + 31) / 32;
  for (int b0 = 0; b0 < A.n_beams; b0 += LIDAR_BEAMS) {
    const int nb = min(LIDAR_BEAMS, A.n_beams - b0);      // beams b0 .. b0 + nb - 1 in this pass
    for (int k = lane; k < nb; k += 32) best[k] = INFINITY;
    if (lane == 0) *cnt = 0;
    __syncwarp();
    // Sources in rounds of 32: the other participants (a cheap centre-distance test first; a box in reach contributes
    // its four ring edges, :146-153), then the map segments (:137-143).  Edges within the range go to the shared chunk
    // with their beam window; the chunk is scanned whenever the next round might not fit.
    for (int r = 0; r < part_rounds + seg_rounds; ++r) {
      if (r < part_rounds) {
        const int j = 1 + r * 32 + lane;
        const int tj = j < A.M ? (int)A.type_id[base + j] : 255;
        if (tj < A.n_types && A.table[tj].shape() == SHAPE_OBB) {
          const Params& pj = A.table[tj];
          const double xj = A.x[base + j], yj = A.y[base + j];
          const double reach = R + (double)pj.rbound * 1.000001 + 1e-6;
          if ((xj - x0) * (xj - x0) + (yj - y0) * (yj - y0) <= reach * reach) {
            double cx[4], cy[4], ex[4], ey[4];
            rect_corners_f64(xj, yj, A.h[base + j], pj.half_len, pj.half_wid, cx, cy);
#pragma unroll
            for (int k = 0; k < 4; ++k) {   // affine [a, b, -b, a, xoff, yoff]
              ex[k] = ca * cx[k] + sa * cy[k] + xoff;
              ey[k] = -sa * cx[k] + ca * cy[k] + yoff;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const double x1 = ex[k], y1 = ey[k], x2 = ex[(k + 1) & 3], y2 = ey[(k + 1) & 3];
              const double d2 = point_segment_dist2(x1, y1, x2, y2);
              if (d2 < R2 * 1.0000001 + 1e-9) {
                const int slot = atomicAdd(cnt, 1);
                edge[slot][0] = x1; edge[slot][1] = y1; edge[slot][2] = x2; edge[slot][3] = y2;
                win[slot] = beam_window(x1, y1, x2, y2, d2, A.n_beams);
              }
            }
          }
        }
      } else {
        const int si = (r - part_rounds) * 32 + lane;
        if (si < n_seg) {
          const float4 sg = seg[si];
          const double x1 = ca * sg.x + sa * sg.y + xoff, y1 = -sa * sg.x + ca * sg.y + yoff;
          const double x2 = ca * sg.z + sa * sg.w + xoff, y2 = -sa * sg.z + ca * sg.w + yoff;
          const double d2 = point_segment_dist2(x1, y1, x2, y2);
          if (d2 < R2 * 1.0000001 + 1e-9) {
            const int slot = atomicAdd(cnt, 1);
            edge[slot][0] = x1; edge[slot][1] = y1; edge[slot][2] = x2; edge[slot][3] = y2;
            win[slot] = beam_window(x1, y1, x2, y2, d2, A.n_beams);
          }
        }
      }
      __syncwarp();
      const int n_e = *cnt;
      if (n_e + 128 <= LIDAR_EDGES && r + 1 < part_rounds + seg_rounds) continue;   // the next round still fits
      // ---- edge by edge, the lanes share the beams of its window (lidar.py:160-213 for those pairs)
      for (int i = 0; i < n_e; ++i) {
        const double x1 = edge[i][0], y1 = edge[i][1], x2 = edge[i][2], y2 = edge[i][3];
        const BeamWindow w = win[i];
        const double d = y2 - y1, e = x1 - x2, f = y1 * x2 - x1 * y2;
        const double xlo = fmin(x1, x2) - 1e-8, xhi = fmax(x1, x2) + 1e-8, ylo = fmin(y1, y2) - 1e-8, yhi = fmax(y1, y2) + 1e-8;
        for (int t = lane; t < w.y; t += 32) {
          int b = w.x + t;
          if (b >= A.n_beams) b -= A.n_beams;
          const int k = b - b0;
          if (k < 0 || k >= nb) continue;
          const double cb = A.beam_cs[2 * b], sb = A.beam_cs[2 * b + 1];
          const double a_ = sb, b_ = -cb;
          const double det = a_ * e - b_ * d;
          if (det != 0.0) {
            const double rx = (b_ * f) / det, ry = (-a_ * f) / det;
            const double lx = cb * R, ly = sb * R;
            const bool okx = !(rx > fmax(1e-8, lx) + 1e-8) && !(rx < fmin(-1e-8, lx) - 1e-8) && !(rx > xhi) && !(rx < xlo);
            const bool oky = !(ry > fmax(1e-8, ly) + 1e-8) && !(ry < fmin(-1e-8, ly) - 1e-8) && !(ry > yhi) && !(ry < ylo);
            if (okx && oky) {
              const double dist = sqrt(rx * rx + ry * ry);
              if (dist < R) best[k] = fminf(best[k], (float)dist);   // clip to the range, range -> inf (:211-213)
            }
          }
        }
        __syncwarp();   // the next edge's window may hand the same beam to another lane
      }
      if (lane == 0) *cnt = 0;
      __syncwarp();
    }
    for (int k = lane; k < nb; k += 32) out[b0 + k] = best[k];
    __syncwarp();
  }
}

// ============================================================================ done exchange over peer memory
// All-gather of the per-rank done masks as ONE small kernel per rank and step, over NVLink / NVSwitch peer memory:
//   put     warp w serves the peers w, w + warps, ...: its lanes store 16-byte pieces of this rank's mask into slot
//           (step % slots), row `rank`, of that peer's gather ring (the own ring included);
//   signal  every lane fences its stores to system scope, the warp synchronises and lane 0 writes step + 1 into word
//           `rank` of the peer's flag array (a strong relaxed store behind the fence = a release): ONE fence round
//           trip per peer, all peers in parallel - not a chain of release stores issued by one thread;
//   wait    lanes 0 .. world-1 of warp 0 poll the OWN flag array (acquire, system scope) until every rank has signalled
//           step - lag; bounded (`timeout` SM cycles): on expiry the sticky error word is set and dst is filled with 0xFF;
//   copy    the slot of step - lag (all ranks' masks in rank order) goes to the caller's array.
// lag = 0 is the synchronous all-gather (the kernel cannot retire before the slowest rank's tick of this step has
// signalled).  lag >= 1 delivers the masks `lag` steps late: by then every signal has long arrived, the wait never spins
// and the kernel is a few microseconds of posted stores - the exchange leaves the critical path (the consumer of the
// gathered masks, a learner or reset scheduler, is behind the simulation anyway).  The kernels of one rank run in
// stream order and kernel k only completes after every rank has signalled step k - lag, i.e. after every rank's kernel
// k - lag - 1 has copied step k - 2 lag - 1 out: a ring of 2 lag + 2 slots is never overwritten before it was read.
struct AllGatherArgs {
  unsigned char* peer[T2D_MAX_RANKS];   // every rank's exchange allocation (own included)
  unsigned char* base;                  // = peer[rank]
  const unsigned char* local;           // this rank's done mask [n_real]
  unsigned char* dst;                   // [world * n_local]
  int world, rank, n_local, n_real, slots, lag;
  long long timeout;                    // SM cycles the wait may spin
};

__global__ void __launch_bounds__(512) t2d_exchange_allgather_kernel(const __grid_constant__ AllGatherArgs A) {
  __shared__ int s_ok;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  const size_t flag_off = (size_t)A.slots * A.world * A.n_local;
  unsigned* words = reinterpret_cast<unsigned*>(A.base + flag_off);      // [0, MAX_RANKS): flags; then step, -, -, error
  const unsigned step = words[T2D_MAX_RANKS];
  const size_t row = (size_t)(step % (unsigned)A.slots) * A.world * A.n_local + (size_t)A.rank * A.n_local;
  if (threadIdx.x == 0) s_ok = 1;
  // ---- put + signal, one warp per peer
  const int n16 = A.n_local / 16;   // n_local is a multiple of 16; the tail beyond n_real is zero
  for (int p = warp; p < A.world; p += warps) {
    uint4* out = reinterpret_cast<uint4*>(A.peer[p] + row);
    for (int i = lane; i < n16; i += 32) {
      uint4 v;
      if (16 * i + 16 <= A.n_real && (reinterpret_cast<uintptr_t>(A.local) & 15) == 0) {
        v = __ldcg(reinterpret_cast<const uint4*>(A.local) + i);
      } else {
        unsigned char b[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) b[k] = (16 * i + k < A.n_real) ? A.local[16 * i + k] : (unsigned char)0;
        memcpy(&v, b, 16);
      }
      out[i] = v;
    }
    __threadfence_system();
    __syncwarp();
    if (lane == 0) {
      unsigned* f = reinterpret_cast<unsigned*>(A.peer[p] + flag_off) + A.rank;
      asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(f), "r"(step + 1u) : "memory");
    }
  }
  // ---- wait for step - lag
  const bool deliver = step >= (unsigned)A.lag;
  const unsigned target = step - (unsigned)A.lag;     // the step whose masks this call delivers
  if (deliver && threadIdx.x < (unsigned)A.world) {
    const unsigned* f = words + threadIdx.x;
    const long long t0 = clock64();
    unsigned v;
    for (;;) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if (v >= target + 1u) break;
      if (clock64() - t0 > A.timeout) { s_ok = 0; break; }
      __nanosleep(20);
    }
  }
  __syncthreads();
  const size_t bytes = (size_t)A.world * A.n_local;
  if (deliver) {
    if (s_ok) {
      // ---- copy
      const unsigned char* src = A.base + (size_t)(target % (unsigned)A.slots) * bytes;
      if ((reinterpret_cast<uintptr_t>(A.dst) & 15) == 0) {
        for (size_t i = threadIdx.x; i < bytes / 16; i += blockDim.x)
          reinterpret_cast<uint4*>(A.dst)[i] = __ldcg(reinterpret_cast<const uint4*>(src) + i);
      } else {
        for (size_t i = threadIdx.x; i < bytes; i += blockDim.x) A.dst[i] = __ldcg(src + i);
      }
    } else {
      // a rank never showed up: the caller must not mistake stale masks for this step's - 0xFF is no done value
      for (size_t i = threadIdx.x; i < bytes; i += blockDim.x) A.dst[i] = (unsigned char)0xFF;
      if (threadIdx.x == 0) words[T2D_MAX_RANKS + 3] = 1u;
    }
  }
  if (threadIdx.x == 0) words[T2D_MAX_RANKS] = step + 1u;
}

// ============================================================================ K5: NPC controllers
// One warp per scenario; lane l owns participants l, l + 32, ... .  fp64 on the fp32 state (a few dozen flops per
// participant: the kernel is bound by its ~30 B / participant of HBM traffic).  All reads of last_accel (own and the
// leader's, previous tick) happen before the warp barrier, all writes (this tick) after it.
struct PathVertex { double x, y, cum, len; };   // vertex, arc length up to it, length of the segment that starts here

struct CtrlArgs {
  const float *x, *y, *h, *v;
  const uint8_t* type_id;
  const Params* table;
  int n_types;
  const t2d_controller_params* ctab;
  int n_ctrl;
  const uint8_t* ctrl_id;
  const int16_t* lead;
  const int16_t* path_id;
  const PathVertex* path_v;
  const int* path_off;
  int n_paths;
  float* last_accel;
  float* action;
  const float* ego_action;   // [N][2] or nullptr: participant 0's action (written into its row of `action` as well)
  int N, M, steer_first;
};

__device__ __forceinline__ double clip_np(double v, double lo, double hi) {   // np.clip: NaN propagates
  return v != v ? v : fmin(fmax(v, lo), hi);
}

// acceleration_controller.py:82-130: cruise, or adaptive cruise when a leader is given
__device__ double longitudinal_law(const t2d_controller_params& p, double v, double x, double y, double a_last, bool has_lead,
                                   double vl, double xl, double yl, double al) {
  const double kp = (double)p.kp;
  double a;
  if (has_lead) {
    const double d_front = sqrt((x - xl) * (x - xl) + (y - yl) * (y - yl));                  // :114
    const double d_target = clip_np(v * (double)p.interval + 5.0, 7.0, 80.0);                // :115-118, :42-45
    const double rel_speed = vl - v;                                                         // :120
    const double rel_target_speed = (d_target - d_front) / kp;                               // :121
    const double rel_accel = (rel_target_speed - rel_speed) / kp;                            // :122
    a = al - rel_accel;                                                                      // :124
  } else {
    a = ((double)p.target_speed - v) / kp;                                                   // :94
  }
  const double w = (double)p.accel_change_rate * (double)p.delta_t;
  a = clip_np(a, a_last - w, a_last + w);                                                    // :95-99, :126-130
  return clip_np(a, (double)p.min_accel, (double)p.max_accel);
}

// (v / v_des) ** delta: the IDM exponent is 4 by default - two multiplications instead of the general pow()
__device__ __forceinline__ double idm_pow(double r, double delta) {
  if (delta == 4.0) { const double r2 = r * r; return r2 * r2; }
  if (delta == 2.0) return r * r;
  return pow(r, delta);
}

// idm_controller.py:59-141
__device__ double idm_law(const t2d_controller_params& p, double v, double x, double y, bool has_lead, double vl, double xl,
                          double yl) {
  const double vd = (double)p.desired_speed, am = (double)p.max_acceleration, b = (double)p.comfortable_deceleration;
  double a;
  if (!has_lead) {
    a = vd > 0.0 ? am * (1.0 - idm_pow(v / vd, (double)p.delta)) : (v > 0.0 ? -b : 0.0);     // :74-82
  } else {
    const double dist = sqrt((xl - x) * (xl - x) + (yl - y) * (yl - y));                     // :107-109 (np.hypot, no overflow concern at map scale)
    const double dv = vl - v;                                                                // :112
    double s_star = (double)p.min_spacing + v * (double)p.time_headway + (v * dv) / (2.0 * sqrt(am * b));   // :116-120
    s_star = fmax(s_star, (double)p.min_spacing);                                            // :121
    if (dist > 0.0) {
      const double ratio = vd > 0.0 ? idm_pow(v / vd, (double)p.delta) : (v > 0.0 ? 1.0 : 0.0);  // :127-130
      const double q = s_star / dist;
      a = am * (1.0 - ratio - q * q);                                                        // :132-134
    } else {
      a = -b;                                                                                // :137
    }
  }
  return clip_np(a, -b, am);                                                                 // :89
}

// pure_pursuit_controller.py:51-74,90-92; LineString.interpolate = arc-length walk from the first vertex
__device__ double pure_pursuit_law(const t2d_controller_params& p, const PathVertex* pv, int n_vert, double v, double x, double y,
                                   double heading) {
  const double d = fmax(v * (double)p.pp_interval, (double)p.min_pre_aiming_distance);     // :90-91
  double px = pv[n_vert - 1].x, py = pv[n_vert - 1].y;
  for (int i = 0; i + 1 < n_vert; ++i) {
    const PathVertex q = pv[i];
    if (d <= q.cum + q.len && q.len > 0.0) {
      const double t = (d - q.cum) / q.len;
      px = q.x + t * (pv[i + 1].x - q.x);
      py = q.y + t * (pv[i + 1].y - q.y);
      break;
    }
  }
  const double ang = atan2(py - y, px - x);                                                 // :62-64
  const double dist = hypot(py - y, px - x);                                                // :65-67
  return atan(2.0 * (double)p.wheel_base * sin(ang - heading) / dist);                      // :68-70
}

__global__ void __launch_bounds__(128) t2d_control_kernel(const __grid_constant__ CtrlArgs A) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; n < A.N; n += warps) {
    const size_t base = (size_t)n * A.M;
    float2 out[4];
    float mag[4];
    bool ctl[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = lane + 32 * j;
      ctl[j] = false;
      mag[j] = 0.0f;
      out[j] = make_float2(0.0f, 0.0f);
      if (m >= A.M) continue;
      const int tid = A.type_id[base + m];
      if (tid >= A.n_types) continue;                  // inactive slot
      const Params& tp = A.table[tid];
      out[j] = reinterpret_cast<const float2*>(A.action)[base + m];
      if (m == 0 && A.ego_action != nullptr) { out[j] = reinterpret_cast<const float2*>(A.ego_action)[n]; ctl[j] = true; }   // row 0 <- the ego's action
      const int cid = A.ctrl_id[base + m];
      if (cid < A.n_ctrl && A.ctab[cid].kind != T2D_CTRL_EXTERNAL) {
        const t2d_controller_params& p = A.ctab[cid];
        const double x = A.x[base + m], y = A.y[base + m], v = A.v[base + m];
        const int li = A.lead ? (int)A.lead[base + m] : -1;
        const bool has = li >= 0 && li < A.M && li != m && A.type_id[base + li] < A.n_types;
        double xl = 0.0, yl = 0.0, vl = 0.0, al = 0.0;
        if (has) {
          xl = A.x[base + li]; yl = A.y[base + li]; vl = A.v[base + li]; al = A.last_accel[base + li];
        }
        double acc, steer = 0.0;
        if (p.kind == T2D_CTRL_IDM) {
          acc = idm_law(p, v, x, y, has, vl, xl, yl);
        } else {
          acc = longitudinal_law(p, v, x, y, (double)A.last_accel[base + m], has, vl, xl, yl, al);
          if (p.kind == T2D_CTRL_PURE_PURSUIT) {
            const int pid = A.path_id ? (int)A.path_id[base + m] : -1;
            if (pid >= 0 && pid < A.n_paths)
              steer = pure_pursuit_law(p, A.path_v + A.path_off[pid], A.path_off[pid + 1] - A.path_off[pid], v, x, y,
                                       (double)A.h[base + m]);
          }
        }
        out[j] = A.steer_first ? make_float2((float)steer, (float)acc) : make_float2((float)acc, (float)steer);
        ctl[j] = true;
      }
      // |a| the physics will apply: single_track_kinematics.py:192 clips to the accel range; point_mass.py takes (ax, ay) as is
      if (tp.model() <= T2D_MODEL_DYNAMICS || tp.model() == T2D_MODEL_DRIFT)
        mag[j] = fabsf(clampf(A.steer_first ? out[j].y : out[j].x, tp.accel_lo, tp.accel_hi));
      else if (tp.model() <= T2D_MODEL_POINTMASS_EULER)
        mag[j] = (float)hypot((double)out[j].x, (double)out[j].y);
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = lane + 32 * j;
      if (m >= A.M) continue;
      if (ctl[j]) reinterpret_cast<float2*>(A.action)[base + m] = out[j];
      A.last_accel[base + m] = mag[j];
    }
  }
}

}  // namespace t2d

// =============================================================================================
// C ABI
// =============================================================================================
using namespace t2d;

static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};
static std::atomic<int> g_exchanges_alive{0};   // peer-memory done exchanges in this process (see StepArgs::prefetch)
static std::mutex g_smem_mutex;
static int g_smem_configured[64][4];   // [device][kernel variant]: dynamic shared memory opted in so far (process-wide)

static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                           \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return fail(T2D_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

struct t2d_exchange {
  int device = 0, world = 0, rank = 0, n_local = 0, slots = 0;
  size_t bytes = 0;
  int n_real = 0;
  int threads = 256;                             // CTA size of the exchange kernel (T2D_EXCHANGE_THREADS, read once at create)
  long long timeout_cycles = 4000000000LL;       // how long a wait may spin (~2 s of SM clocks; T2D_EXCHANGE_TIMEOUT_MS)
  unsigned char* base = nullptr;                 // slots x world x n_local done bytes | MAX_RANKS flag words | step, -, -, error
  unsigned char* peer[T2D_MAX_RANKS] = {};       // every rank's base (own included), valid after t2d_exchange_connect
  bool connected = false;
  size_t flag_off() const { return (size_t)slots * world * n_local; }
  unsigned* word(int i) const { return reinterpret_cast<unsigned*>(base + flag_off()) + T2D_MAX_RANKS + i; }   // 0 steps done, 3 error
};

struct t2d_ctx {
  int device = 0, N = 0, M = 0, G = 0, ppl = 4;
  t2d_config cfg{};
  int n_types = 0;
  bool has_pointmass = false;
  bool has_drift = false;
  bool kin_only = false;
  float *wheel_f = nullptr, *wheel_r = nullptr;
  const float *reset_pool_wf = nullptr, *reset_pool_wr = nullptr;   // t2d_bind_reset_wheel_pool
  Params* d_table = nullptr;
  unsigned char* d_map = nullptr;
  uint32_t* d_tile_off = nullptr;   // [n_tiles] byte offsets of the tiles inside d_map
  const uint16_t* tile_id = nullptr;   // caller-owned DEVICE [N] (more than one tile)
  int n_tiles = 0;
  bool has_segments = false;
  MapHeader mh{};
  int map_bytes = 0;
  bool has_bounds = false;
  float bounds[4] = {0, 0, 0, 0};
  float *x = nullptr, *y = nullptr, *h = nullptr, *v = nullptr, *vx = nullptr, *vy = nullptr;
  const uint8_t* type_id = nullptr;
  int32_t* step_count = nullptr;
  int sm_count = 148;
  int max_smem_optin = 0;
  float rb_max = 0.0f;
  const float* ego_action = nullptr;   // t2d_set_ego_action
  const float* goal_target = nullptr;
  float* goal_iou = nullptr;
  float* goal_last_pose = nullptr;
  int32_t* goal_noact_count = nullptr;
  float goal_threshold = 0.95f;
  int goal_noact_max = 0;
  bool use_pdl = true;             // T2D_PDL=0 disables programmatic dependent launch
  int prefetch_override = -1;      // T2D_PREFETCH=0 / 1 (experiments; -1 = on unless a done exchange is alive)
  int wpc_override = 0;            // T2D_WPC=w: warps per CTA of the tick (experiments; 0 = pick from the batch size)
  int grid_limit = 0;              // T2D_GRID_LIMIT=k: at most k CTAs of the persistent tick grid per SM (experiments; 0 = occupancy)
  long long* dbg_clock = nullptr;
  int occ_smem[9] = {-1, -1, -1, -1, -1, -1, -1, -1, -1};   // per warps-per-CTA: smem the cached occupancy was computed for
  int occ_val[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int occ_variant[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  // NPC controllers (t2d_set_controllers / t2d_set_paths / t2d_control)
  t2d_controller_params* d_ctab = nullptr;
  int n_ctrl = 0;
  const uint8_t* ctrl_id = nullptr;
  const int16_t* ctrl_lead = nullptr;
  const int16_t* ctrl_path = nullptr;
  float* ctrl_last_accel = nullptr;
  PathVertex* d_path_v = nullptr;
  int* d_path_off = nullptr;
  int n_paths = 0;
  // t2d_step_host: device staging for the host-resident action / status / done, the copy stream and its events
  static constexpr int MAX_HOST_CHUNKS = 8;
  float* hs_action = nullptr;          // [N][M][2]
  float* hs_ego_pinned = nullptr;      // [N][2] pinned + mapped host staging of the ego actions (t2d_step_host_ego) ...
  const float* hs_ego_dev = nullptr;   // ... and its device-side address: the kernels read it over PCIe, no copy engine involved
  uint8_t* hs_out = nullptr;           // [2][N] status, done
  uint8_t* hs_out_pinned = nullptr;    // pinned host mirror of hs_out
  cudaStream_t hs_copy = nullptr;
  cudaEvent_t hs_begin = nullptr, hs_chunk[MAX_HOST_CHUNKS] = {};
  int host_chunks = 0;                 // 0 = pick from the batch size
};

extern "C" {

int t2d_version(void) { return T2D_VERSION; }
const char* t2d_last_error(void) { return g_err.c_str(); }
int64_t t2d_launch_count(void) { return (int64_t)g_launches.load(); }

static int check_cfg(const t2d_config* cfg) {
  if (!cfg) return fail(T2D_E_INVALID, "cfg is NULL");
  if (cfg->interval_ms <= 0) return fail(T2D_E_INVALID, "interval_ms must be > 0");
  if (cfg->delta_t_ms <= 0) return fail(T2D_E_INVALID, "delta_t_ms must be > 0");
  return T2D_OK;
}

int t2d_create(t2d_ctx** out, int device, int n_scenarios, int m_participants, const t2d_config* cfg) {
  if (!out) return fail(T2D_E_INVALID, "out is NULL");
  *out = nullptr;
  if (int r = check_cfg(cfg)) return r;
  if (n_scenarios <= 0 || m_participants <= 0) return fail(T2D_E_INVALID, "n_scenarios and m_participants must be > 0");
  if (m_participants > T2D_MAX_PARTICIPANTS)
    return fail(T2D_E_UNSUPPORTED, "m_participants > 128: a scenario must fit one warp (4 participants per lane)");
  int count = 0;
  CUDA_TRY(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail(T2D_E_INVALID, "no such CUDA device");
  CUDA_TRY(cudaSetDevice(device));
  t2d_ctx* c = new t2d_ctx();
  c->device = device;
  c->N = n_scenarios;
  c->M = m_participants;
  // participants per lane: 4 (2 was measured on B200 at 4096 x 64 in both rounds: 55 % more instructions, 21.5 vs 13.9 us)
  const int ppl = 4;
  c->ppl = ppl;
  if (const char* e = getenv("T2D_PDL")) c->use_pdl = atoi(e) != 0;
  if (const char* e = getenv("T2D_GRID_LIMIT")) c->grid_limit = std::max(0, atoi(e));
  if (const char* e = getenv("T2D_PREFETCH")) c->prefetch_override = atoi(e) != 0 ? 1 : 0;
  if (const char* e = getenv("T2D_WPC")) {
    const int v = atoi(e);
    if (v >= 1 && v <= MAX_WARPS_PER_CTA) c->wpc_override = v;
  }
  if (const char* e = getenv("T2D_HOST_CHUNKS")) c->host_chunks = std::max(0, std::min(atoi(e), (int)t2d_ctx::MAX_HOST_CHUNKS));
  int g = 1;
  while (g * ppl < m_participants) g <<= 1;
  c->G = g;
  c->cfg = *cfg;
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  c->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  *out = c;
  return T2D_OK;
}

int t2d_destroy(t2d_ctx* c) {
  if (!c) return T2D_OK;
  cudaSetDevice(c->device);
  if (c->d_table) cudaFree(c->d_table);
  if (c->d_map) cudaFree(c->d_map);
  if (c->d_tile_off) cudaFree(c->d_tile_off);
  if (c->d_ctab) cudaFree(c->d_ctab);
  if (c->d_path_v) cudaFree(c->d_path_v);
  if (c->d_path_off) cudaFree(c->d_path_off);
  if (c->hs_action) cudaFree(c->hs_action);
  if (c->hs_ego_pinned) cudaFreeHost(c->hs_ego_pinned);
  if (c->hs_out) cudaFree(c->hs_out);
  if (c->hs_out_pinned) cudaFreeHost(c->hs_out_pinned);
  if (c->hs_begin) cudaEventDestroy(c->hs_begin);
  for (cudaEvent_t e : c->hs_chunk)
    if (e) cudaEventDestroy(e);
  if (c->hs_copy) cudaStreamDestroy(c->hs_copy);
  delete c;
  return T2D_OK;
}

int t2d_set_config(t2d_ctx* c, const t2d_config* cfg) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (int r = check_cfg(cfg)) return r;
  c->cfg = *cfg;
  return T2D_OK;
}

int t2d_set_type_table(t2d_ctx* c, const t2d_type_params* table, int n_types) {
  if (!c || !table) return fail(T2D_E_INVALID, "ctx/table is NULL");
  if (n_types <= 0 || n_types > T2D_MAX_TYPES) return fail(T2D_E_INVALID, "n_types must be in 1..64");
  static_assert(sizeof(t2d_type_params) == sizeof(AbiParams), "type table layout");
  c->has_pointmass = false;
  bool has_drift = false;
  float rb_max = 0.0f;
  for (int i = 0; i < n_types; ++i) {
    const t2d_type_params& p = table[i];
    if (p.shape == T2D_SHAPE_OBB) rb_max = std::max(rb_max, sqrtf(p.half_len * p.half_len + p.half_wid * p.half_wid) * 1.000002f);
    if (p.shape == T2D_SHAPE_CIRCLE) rb_max = std::max(rb_max, p.radius);
    if (p.model < 0 || p.model > T2D_MODEL_DRIFT) return fail(T2D_E_INVALID, "type table: unknown model id");
    if (p.shape < 0 || p.shape > T2D_SHAPE_NONE) return fail(T2D_E_INVALID, "type table: unknown shape id");
    const bool bicycle = p.model <= T2D_MODEL_DYNAMICS || p.model == T2D_MODEL_DRIFT;
    if (bicycle && !(p.lf + p.lr > 0.0f)) return fail(T2D_E_INVALID, "type table: lf + lr must be > 0");
    if (p.model == T2D_MODEL_DYNAMICS && !(p.lf > 0.0f && p.I_z > 0.0f))
      return fail(T2D_E_INVALID, "type table: dynamics needs lf > 0 and I_z > 0");
    if (p.model == T2D_MODEL_DRIFT && !(p.lf > 0.0f && p.I_z > 0.0f && p.mass > 0.0f && p.wheel_radius > 0.0f && p.I_yw > 0.0f))
      return fail(T2D_E_INVALID, "type table: drift needs lf, I_z, mass, wheel_radius and I_yw > 0");
    if (p.model == T2D_MODEL_DRIFT) has_drift = true;
    if (p.shape == T2D_SHAPE_OBB && !(p.half_len >= 0.0f && p.half_wid >= 0.0f))
      return fail(T2D_E_INVALID, "type table: negative OBB half extent");
    if (p.shape == T2D_SHAPE_CIRCLE && !(p.radius >= 0.0f)) return fail(T2D_E_INVALID, "type table: negative radius");
    if (p.model == T2D_MODEL_POINTMASS_NEWTON || p.model == T2D_MODEL_POINTMASS_EULER) c->has_pointmass = true;
  }
  CUDA_TRY(cudaSetDevice(c->device));
  if (!c->d_table) CUDA_TRY(cudaMalloc(&c->d_table, (T2D_MAX_TYPES + 1) * sizeof(Params)));
  {
    std::vector<Params> rows(n_types + 1);
    for (int i = 0; i < n_types; ++i) {
      AbiParams a;
      memcpy(&a, &table[i], sizeof(AbiParams));
      rows[i] = derive_params(a);
    }
    {
      // row n_types: the neutral kinematic row that K1's packed loop gives to slots holding another model or nothing
      // (zero speed and action in, unbounded ranges: every product stays finite and the result is discarded)
      AbiParams a{};
      a.lf = 1.0f; a.lr = 1.0f;
      a.steer_lo = a.speed_lo = a.accel_lo = -INFINITY;
      a.steer_hi = a.speed_hi = a.accel_hi = INFINITY;
      a.model = MODEL_KINEMATICS; a.shape = SHAPE_NONE;
      rows[n_types] = derive_params(a);
    }
    CUDA_TRY(cudaMemcpy(c->d_table, rows.data(), (n_types + 1) * sizeof(Params), cudaMemcpyHostToDevice));
  }
  c->n_types = n_types;
  c->has_drift = has_drift;
  c->rb_max = rb_max;
  c->kin_only = true;
  for (int i = 0; i < n_types; ++i)
    if (table[i].model != T2D_MODEL_KINEMATICS && table[i].model != T2D_MODEL_STATIC) c->kin_only = false;
  for (int w = 0; w < 9; ++w) c->occ_smem[w] = -1;
  return T2D_OK;
}

int t2d_set_map_table(t2d_ctx* c, const t2d_map_tile* tiles, int n_tiles, const uint16_t* tile_id, float cell_size) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (n_tiles < 0 || n_tiles > T2D_MAX_TILES) return fail(T2D_E_INVALID, "n_tiles must be in 0..T2D_MAX_TILES");
  if (n_tiles > 0 && !tiles) return fail(T2D_E_INVALID, "tiles is NULL");
  if (n_tiles > 1 && !tile_id) return fail(T2D_E_INVALID, "tile_id is NULL (needed with more than one tile)");
  // compiled before the current map is released: a rejected table leaves the current map in force
  std::vector<unsigned char> all;
  std::vector<uint32_t> offs;
  std::string err;
  if (int r = compile_map_table(tiles, n_tiles, cell_size, c->rb_max, all, offs, err)) return fail(r, err);
  CUDA_TRY(cudaSetDevice(c->device));
  if (c->d_map) { cudaFree(c->d_map); c->d_map = nullptr; }
  if (c->d_tile_off) { cudaFree(c->d_tile_off); c->d_tile_off = nullptr; }
  c->map_bytes = 0; c->n_tiles = 0; c->tile_id = nullptr; c->has_bounds = false; c->has_segments = false;
  c->mh = MapHeader{};
  if (n_tiles == 0) return T2D_OK;
  bool any_bounds = false, any_seg = false;
  for (int i = 0; i < n_tiles; ++i) {
    any_bounds = any_bounds || tiles[i].bounds != nullptr;
    any_seg = any_seg || tiles[i].n_seg > 0;
  }
  memcpy(&c->mh, all.data(), sizeof(MapHeader));   // tile 0 starts at offset 0
  CUDA_TRY(cudaMalloc(&c->d_map, all.size()));
  CUDA_TRY(cudaMemcpy(c->d_map, all.data(), all.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMalloc(&c->d_tile_off, sizeof(uint32_t) * (size_t)n_tiles));
  CUDA_TRY(cudaMemcpy(c->d_tile_off, offs.data(), sizeof(uint32_t) * (size_t)n_tiles, cudaMemcpyHostToDevice));
  c->n_tiles = n_tiles;
  c->tile_id = n_tiles > 1 ? tile_id : nullptr;
  c->map_bytes = (int)c->mh.smem_bytes;     // what a single tile stages into shared memory
  c->has_bounds = any_bounds; c->has_segments = any_seg;
  if (c->mh.has_bounds) { c->bounds[0] = c->mh.bxmin; c->bounds[1] = c->mh.bxmax; c->bounds[2] = c->mh.bymin; c->bounds[3] = c->mh.bymax; }
  return T2D_OK;
}

int t2d_set_map_polygons(t2d_ctx* c, const float* segments, int n_seg, const int32_t* poly_start, int n_poly, const float* bounds,
                         float cell_size) {
  if (n_seg == 0 && !bounds) return t2d_set_map_table(c, nullptr, 0, nullptr, cell_size);
  t2d_map_tile t{};
  t.segments = segments; t.n_seg = n_seg; t.poly_start = poly_start; t.n_poly = n_poly; t.bounds = bounds;
  return t2d_set_map_table(c, &t, 1, nullptr, cell_size);
}

int t2d_set_map(t2d_ctx* c, const float* segments, int n_seg, const float* bounds, float cell_size) {
  return t2d_set_map_polygons(c, segments, n_seg, nullptr, 0, bounds, cell_size);
}

int t2d_bind_state(t2d_ctx* c, float* x, float* y, float* heading, float* speed, float* vx, float* vy,
                   const uint8_t* type_id, int32_t* step_count) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!x || !y || !heading || !speed || !vx || !vy || !type_id || !step_count)
    return fail(T2D_E_INVALID, "t2d_bind_state: NULL array");
  c->x = x; c->y = y; c->h = heading; c->v = speed; c->vx = vx; c->vy = vy;
  c->type_id = type_id; c->step_count = step_count;
  return T2D_OK;
}

int t2d_bind_wheel_state(t2d_ctx* c, float* omega_front, float* omega_rear) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if ((omega_front == nullptr) != (omega_rear == nullptr)) return fail(T2D_E_INVALID, "t2d_bind_wheel_state: one array is NULL");
  c->wheel_f = omega_front; c->wheel_r = omega_rear;
  return T2D_OK;
}

int t2d_bind_reset_wheel_pool(t2d_ctx* c, const float* pool_omega_front, const float* pool_omega_rear) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if ((pool_omega_front == nullptr) != (pool_omega_rear == nullptr)) return fail(T2D_E_INVALID, "t2d_bind_reset_wheel_pool: one array is NULL");
  c->reset_pool_wf = pool_omega_front; c->reset_pool_wr = pool_omega_rear;
  return T2D_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Warps per CTA of the tick.  One wave (the usual case: every warp tile is resident at once and the kernel's duration is
// one tile's lifetime): the SM with the most warps sets the pace, and every CTA costs a launch + prologue (barrier
// init, TMA staging) - measured on B200 at 4096 x 64: ~0.19 us per extra warp on the fullest SM, ~0.08 us per CTA on it
// (2 x 7 warps: 16.4 us, 7 x 2: 16.8 us, 3 x 5: 16.7 us, 2 x 8: 17.0 us, 3 x 6 - a second wave at 128 registers - 23.9 us;
// 1-warp CTAs are far worse and are not considered).  Several waves: persistent CTAs of the largest size.
static int pick_wpc(long long tiles, int sm_count) {
  const int resident_warps = 14;   // per SM at the kernel's register budget, rounded down to what every variant reaches
  if (tiles > (long long)sm_count * resident_warps) return MAX_WARPS_PER_CTA;
  int best = 2;
  double best_cost = 1e30;
  for (int w = 2; w <= MAX_WARPS_PER_CTA; ++w) {
    const long long ctas = (tiles + w - 1) / w;
    const long long per_sm = (ctas + sm_count - 1) / sm_count;
    const double cost = (double)(per_sm * w) + 0.42 * (double)per_sm;
    if (cost < best_cost - 1e-9 || (cost < best_cost + 1e-9 && w > best)) { best_cost = cost; best = w; }
  }
  return best;
}

// Launches K1 over the scenarios [first, first + count) of the bound state; the per-participant / per-scenario
// pointers passed in (action, flags, ..., done) address scenario `first` already.
static int launch_step(t2d_ctx* c, const float* action, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment,
                       uint8_t* scn_status, uint8_t* done, void* stream, int do_physics, int first = 0, int count = -1) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!c->x) return fail(T2D_E_STATE, "state not bound: call t2d_bind_state first");
  if (!c->d_table || c->n_types == 0) return fail(T2D_E_STATE, "type table not set: call t2d_set_type_table first");
  if (do_physics && !action) return fail(T2D_E_INVALID, "action is NULL");
  if (do_physics && c->has_drift && !(c->wheel_f && c->wheel_r))
    return fail(T2D_E_STATE, "the type table holds a SingleTrackDrift row: call t2d_bind_wheel_state first");
  CUDA_TRY(cudaSetDevice(c->device));
  if (count < 0) count = c->N - first;
  if (first < 0 || count <= 0 || first + count > c->N) return fail(T2D_E_INVALID, "scenario range out of bounds");
  const size_t p0 = (size_t)first * c->M;
  StepArgs A{};
  A.x = c->x + p0; A.y = c->y + p0; A.h = c->h + p0; A.v = c->v + p0; A.vx = c->vx + p0; A.vy = c->vy + p0;
  A.type_id = c->type_id + p0; A.step_count = c->step_count + first;
  A.wheel_f = c->wheel_f ? c->wheel_f + p0 : nullptr; A.wheel_r = c->wheel_r ? c->wheel_r + p0 : nullptr;
  A.action = action; A.ego_action = c->ego_action ? c->ego_action + 2 * (size_t)first : nullptr; A.flags = flags; A.hit_index = hit_index; A.hit_segment = hit_segment;
  A.scn_status = scn_status; A.done = done;
  const bool map_table = c->n_tiles > 1;
  A.map_blob = c->d_map; A.map_bytes = c->map_bytes; A.mh = c->mh;
  A.tile_off = c->d_tile_off; A.tile_id = map_table ? c->tile_id + first : nullptr;
  A.map_in_smem = (!map_table && c->d_map && c->mh.n_seg > 0 && c->map_bytes <= MAP_SMEM_LIMIT) ? 1 : 0;
  A.table = c->d_table; A.n_types = c->n_types;
  A.N = count; A.M = c->M; A.G = c->G;
  const int delta_t = std::min(c->cfg.delta_t_ms, c->cfg.interval_ms);
  A.n_steps = c->cfg.interval_ms / delta_t;                       // single_track_kinematics.py:129
  A.dt = (float)((double)delta_t / 1000.0);                      // :128
  A.dt_rem = (float)((double)(c->cfg.interval_ms % delta_t) / 1000.0);   // :130,152
  A.dt_d = (double)delta_t / 1000.0;
  A.dt_rem_d = (double)(c->cfg.interval_ms % delta_t) / 1000.0;
  A.interval_d = (double)c->cfg.interval_ms / 1000.0;                  // point_mass.py:86
  A.max_step = c->cfg.max_step; A.cfg_flags = c->cfg.flags;
  A.do_physics = do_physics; A.has_bounds = c->has_bounds ? 1 : 0;
  A.bxmin = c->bounds[0]; A.bxmax = c->bounds[1]; A.bymin = c->bounds[2]; A.bymax = c->bounds[3];
  A.prefetch = c->prefetch_override >= 0 ? c->prefetch_override : (g_exchanges_alive.load() == 0 ? 1 : 0);
  A.needs_vel_in = (c->has_pointmass || c->has_drift) ? 1 : 0;   // (drift: K1 passes the pre-pass's vx, vy through)
  bool vec = (c->M % c->ppl == 0) && aligned16(A.x) && aligned16(A.y) && aligned16(A.h) && aligned16(A.v) && aligned16(A.vx) &&
             aligned16(A.vy) && (reinterpret_cast<uintptr_t>(A.type_id) % 4 == 0) && (!action || aligned16(action)) &&
             (!flags || reinterpret_cast<uintptr_t>(flags) % 4 == 0) && (!hit_index || reinterpret_cast<uintptr_t>(hit_index) % 8 == 0) &&
             (!hit_segment || reinterpret_cast<uintptr_t>(hit_segment) % 8 == 0);
  A.vec_ok = vec ? 1 : 0;

  A.rb_max = c->rb_max;
  A.dbg_clock = c->dbg_clock;
  A.goal_target = c->goal_target ? c->goal_target + 5 * (size_t)first : nullptr;
  A.goal_iou = c->goal_iou ? c->goal_iou + first : nullptr;
  A.goal_last_pose = c->goal_last_pose ? c->goal_last_pose + 4 * (size_t)first : nullptr;
  A.goal_noact_count = c->goal_noact_count ? c->goal_noact_count + first : nullptr; A.goal_threshold = c->goal_threshold; A.goal_noact_max = c->goal_noact_max;
  const int table_bytes = (((c->n_types + 1) * (int)sizeof(Params) + 15) / 16) * 16;   // + the neutral row
  const int spw = 32 / c->G;
  const long long tiles = ((long long)count + spw - 1) / spw;
  int wpc = pick_wpc(tiles, c->sm_count);
  if (c->wpc_override > 0) wpc = c->wpc_override;   // T2D_WPC (experiments), read once at t2d_create
  {
    int off = (A.map_in_smem ? A.map_bytes : 0) + table_bytes;
    A.off_poseA = off; off += wpc * POSE_PER_WARP * (int)sizeof(float4);
    A.off_poseB = off; off += wpc * POSE_PER_WARP * (int)sizeof(float4);
    A.off_hit = off; off += wpc * POSE_PER_WARP * (int)sizeof(int);
    A.off_queue = off; off += wpc * QCAP * 4;
    A.off_posx = off; off += wpc * POS_EXT_PER_WARP * 4;
    A.off_posy = off; off += wpc * POS_EXT_PER_WARP * 4;
    A.off_qcount = off; off += ((wpc + 3) & ~3) * 4;
    A.off_bar = off; off += 16;
    A.wpc = wpc;
    A.table_bytes = table_bytes;
    A.n_tiles = (int)tiles;
    A.g_shift = 0;
    while ((1 << A.g_shift) < c->G) ++A.g_shift;
    const int MP = c->G * c->ppl;
    A.mp_shift = 0;
    while ((1 << A.mp_shift) < MP) ++A.mp_shift;
    A.ext = ((3 * MP) / 2 + 16 + 3) & ~3;   // a multiple of 4 floats: every scenario's window starts 16-byte aligned
  }
  const int smem = A.off_bar + 16;
  if (smem > c->max_smem_optin) return fail(T2D_E_UNSUPPORTED, "shared memory budget exceeded");
  using kernel_t = void (*)(StepArgs);
  kernel_t kern;
  if (c->kin_only) kern = map_table ? (kernel_t)t2d_step_kernel<4, true, true> : (kernel_t)t2d_step_kernel<4, true, false>;
  else kern = map_table ? (kernel_t)t2d_step_kernel<4, false, true> : (kernel_t)t2d_step_kernel<4, false, false>;
  {
    // cudaFuncSetAttribute applies to the kernel function for the whole process and SETS the value: worlds of
    // different sizes share it, so the opt-in is tracked per (device, kernel variant) and only ever raised.
    const int variant = (c->kin_only ? 2 : 0) + (map_table ? 1 : 0);
    std::lock_guard<std::mutex> lock(g_smem_mutex);
    int& configured = g_smem_configured[c->device % 64][variant];
    if (smem > configured) {
      CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      configured = smem;
    }
  }
  if (do_physics && c->has_drift) {
    const long long total = (long long)count * c->M;
    const int dgrid = (int)std::min<long long>((total + 127) / 128, (long long)c->sm_count * 16);
    t2d_drift_kernel<<<dgrid, 128, 0, (cudaStream_t)stream>>>(A);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
  }
  const long long ctas_needed = (tiles + wpc - 1) / wpc;
  if (c->occ_smem[wpc] != smem || c->occ_variant[wpc] != (map_table ? 1 : 0)) {
    int per_sm = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, wpc * 32, smem));
    c->occ_val[wpc] = per_sm < 1 ? 1 : per_sm;
    c->occ_smem[wpc] = smem;
    c->occ_variant[wpc] = map_table ? 1 : 0;
  }
  int per_sm_ctas = c->occ_val[wpc];
  if (c->grid_limit > 0) per_sm_ctas = std::min(per_sm_ctas, c->grid_limit);   // T2D_GRID_LIMIT: leave CTA slots to other streams
  const long long resident = (long long)c->sm_count * per_sm_ctas;
  const int grid = (int)std::max(1LL, std::min(ctas_needed, resident));
  {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)(wpc * 32));
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = c->use_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, A));
  }
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

int t2d_set_goal(t2d_ctx* c, const float* target, float arrival_threshold, int no_action_max_step, float* iou_out, float* last_pose,
                 int32_t* no_action_count) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (target && (!iou_out || !last_pose || !no_action_count)) return fail(T2D_E_INVALID, "t2d_set_goal: NULL output array");
  if (target && !(arrival_threshold > 0.0f && arrival_threshold <= 1.0f)) return fail(T2D_E_INVALID, "arrival_threshold must be in (0, 1]");
  c->goal_target = target; c->goal_iou = iou_out; c->goal_last_pose = last_pose; c->goal_noact_count = no_action_count;
  c->goal_threshold = arrival_threshold; c->goal_noact_max = no_action_max_step;
  return T2D_OK;
}

int t2d_debug_set_clock_buffer(t2d_ctx* c, long long* device_buffer) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  c->dbg_clock = device_buffer;
  return T2D_OK;
}

int t2d_step(t2d_ctx* c, const float* action, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment, uint8_t* scn_status,
             uint8_t* done, void* stream) {
  return launch_step(c, action, flags, hit_index, hit_segment, scn_status, done, stream, 1);
}

int t2d_step_host(t2d_ctx* c, const float* action_host, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment,
                  uint8_t* scn_status_host, uint8_t* done_host, void* stream) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!action_host) return fail(T2D_E_INVALID, "action is NULL");
  CUDA_TRY(cudaSetDevice(c->device));
  const int N = c->N, M = c->M;
  if (!c->hs_action) {
    CUDA_TRY(cudaMalloc(&c->hs_action, (size_t)N * M * 2 * sizeof(float)));
    CUDA_TRY(cudaMalloc(&c->hs_out, 2 * (size_t)N));
    CUDA_TRY(cudaMallocHost(&c->hs_out_pinned, 2 * (size_t)N));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->hs_copy, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&c->hs_begin, cudaEventDisableTiming));
    for (cudaEvent_t& e : c->hs_chunk) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  // Chunks of whole scenarios: the copy of chunk k + 1 (copy engine, own stream) runs under the kernel of chunk k.
  // Measured on B200 (profiles/r01_e2e_probe.txt): at 4096 x 64 the 2 MiB upload is ~50 us against a 21 us kernel
  // whose duration is one tile's lifetime whatever the batch, so splitting only adds ~3.5 us per chunk; it pays
  // once a chunk alone fills the GPU, i.e. from ~1 M participants (8 MiB of actions) per chunk upwards.
  int chunks = c->host_chunks;
  if (chunks <= 0) chunks = (int)std::min<long long>(t2d_ctx::MAX_HOST_CHUNKS, std::max<long long>(1, (long long)N * M / (1 << 20)));
  int per = (N + chunks - 1) / chunks;
  per = (per + 31) & ~31;   // whole warp tiles (<= 32 scenarios per warp): a chunked tick groups lanes exactly as t2d_step does
  cudaStream_t s = (cudaStream_t)stream;
  const bool split = per < N;   // a single chunk needs no second stream
  if (split) {
    CUDA_TRY(cudaEventRecord(c->hs_begin, s));            // the copies follow whatever the caller queued on `stream`
    CUDA_TRY(cudaStreamWaitEvent(c->hs_copy, c->hs_begin, 0));
  }
  int k = 0;
  for (int first = 0; first < N; first += per, ++k) {
    const int count = std::min(per, N - first);
    const size_t a0 = (size_t)first * M * 2;
    CUDA_TRY(cudaMemcpyAsync(c->hs_action + a0, action_host + a0, (size_t)count * M * 2 * sizeof(float), cudaMemcpyHostToDevice,
                             split ? c->hs_copy : s));
    if (split) {
      CUDA_TRY(cudaEventRecord(c->hs_chunk[k], c->hs_copy));
      CUDA_TRY(cudaStreamWaitEvent(s, c->hs_chunk[k], 0));
    }
    const size_t p0 = (size_t)first * M;
    if (int r = launch_step(c, c->hs_action + a0, flags ? flags + p0 : nullptr, hit_index ? hit_index + p0 : nullptr,
                            hit_segment ? hit_segment + p0 : nullptr, c->hs_out + first, c->hs_out + N + first, stream, 1, first, count))
      return r;
  }
  CUDA_TRY(cudaMemcpyAsync(c->hs_out_pinned, c->hs_out, 2 * (size_t)N, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  if (scn_status_host) memcpy(scn_status_host, c->hs_out_pinned, (size_t)N);
  if (done_host) memcpy(done_host, c->hs_out_pinned + N, (size_t)N);
  return T2D_OK;
}

int t2d_set_prefetch(t2d_ctx* c, int mode) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (mode < -1 || mode > 1) return fail(T2D_E_INVALID, "prefetch mode must be -1 (policy), 0 (off) or 1 (on)");
  c->prefetch_override = mode;
  return T2D_OK;
}

int t2d_set_ego_action(t2d_ctx* c, const float* ego_action) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (ego_action && reinterpret_cast<uintptr_t>(ego_action) % 8 != 0) return fail(T2D_E_INVALID, "ego_action must be 8-byte aligned");
  c->ego_action = ego_action;
  return T2D_OK;
}

int t2d_step_host_ego(t2d_ctx* c, const float* ego_action_host, float* action, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment,
                      uint8_t* scn_status_host, uint8_t* done_host, void* stream) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!ego_action_host || !action) return fail(T2D_E_INVALID, "ego_action / action is NULL");
  CUDA_TRY(cudaSetDevice(c->device));
  const int N = c->N;
  if (!c->hs_ego_pinned) {
    // pinned AND mapped: the first kernel of the step reads the 8 N bytes straight from host memory (one PCIe round trip
    // inside the kernel) instead of waiting for a copy-engine transfer and the stream dependency behind it
    CUDA_TRY(cudaHostAlloc(&c->hs_ego_pinned, (size_t)N * 2 * sizeof(float), cudaHostAllocMapped));
    float* dev = nullptr;
    CUDA_TRY(cudaHostGetDevicePointer(&dev, c->hs_ego_pinned, 0));
    c->hs_ego_dev = dev;
  }
  if (!c->hs_out) {
    CUDA_TRY(cudaMalloc(&c->hs_out, 2 * (size_t)N));
    CUDA_TRY(cudaMallocHost(&c->hs_out_pinned, 2 * (size_t)N));
  }
  cudaStream_t s = (cudaStream_t)stream;
  memcpy(c->hs_ego_pinned, ego_action_host, (size_t)N * 2 * sizeof(float));
  const float* saved = c->ego_action;
  int r = T2D_OK;
  if (c->d_ctab) {
    // the controllers' launch fetches the ego actions and writes them into row 0 of `action`; the other participants'
    // actions never leave the device; the tick then reads everything from `action`
    c->ego_action = c->hs_ego_dev;
    r = t2d_control(c, action, stream);
    c->ego_action = nullptr;
  } else {
    c->ego_action = c->hs_ego_dev;
  }
  if (r == T2D_OK) r = launch_step(c, action, flags, hit_index, hit_segment, c->hs_out, c->hs_out + N, stream, 1);
  c->ego_action = saved;
  if (r != T2D_OK) return r;
  CUDA_TRY(cudaMemcpyAsync(c->hs_out_pinned, c->hs_out, 2 * (size_t)N, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  if (scn_status_host) memcpy(scn_status_host, c->hs_out_pinned, (size_t)N);
  if (done_host) memcpy(done_host, c->hs_out_pinned + N, (size_t)N);
  return T2D_OK;
}

int t2d_env_epilogue(t2d_ctx* c, const uint8_t* flags, const uint8_t* scn_status, float* reward, uint8_t* terminated,
                     uint8_t* truncated, uint8_t* traffic_status, uint8_t* done, float* max_iou, float* min_dist,
                     int reset_trackers_on_done, void* stream) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!c->x) return fail(T2D_E_STATE, "state not bound: call t2d_bind_state first");
  if (!flags || !scn_status || !reward) return fail(T2D_E_INVALID, "t2d_env_epilogue: flags / scn_status / reward is NULL");
  CUDA_TRY(cudaSetDevice(c->device));
  EnvArgs A{};
  A.flags = flags; A.status = scn_status; A.step_count = c->step_count; A.x = c->x; A.y = c->y;
  A.iou = c->goal_target ? c->goal_iou : nullptr; A.target = c->goal_target;
  A.max_iou = max_iou; A.min_dist = min_dist;
  A.reward = reward; A.terminated = terminated; A.truncated = truncated; A.done = done; A.traffic_status = traffic_status;
  A.N = c->N; A.M = c->M; A.max_step = c->cfg.max_step; A.reset_trackers = reset_trackers_on_done ? 1 : 0;
  const long long total = (long long)c->N * c->M;
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)c->sm_count * 8);
  t2d_env_epilogue_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

int t2d_check_events(t2d_ctx* c, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment, void* stream) {
  return launch_step(c, nullptr, flags, hit_index, hit_segment, nullptr, nullptr, stream, 0);
}

int t2d_reset(t2d_ctx* c, const uint8_t* mask, const int32_t* pool_index, int n_pool, const float* pool_x, const float* pool_y,
              const float* pool_heading, const float* pool_speed, const float* pool_vx, const float* pool_vy, void* stream) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!c->x) return fail(T2D_E_STATE, "state not bound: call t2d_bind_state first");
  if (!mask || !pool_x || !pool_y || !pool_heading || !pool_speed) return fail(T2D_E_INVALID, "t2d_reset: NULL array");
  if (n_pool <= 0) return fail(T2D_E_INVALID, "n_pool must be > 0");
  CUDA_TRY(cudaSetDevice(c->device));
  ResetArgs A{};
  A.x = c->x; A.y = c->y; A.h = c->h; A.v = c->v; A.vx = c->vx; A.vy = c->vy; A.step_count = c->step_count;
  A.mask = mask; A.pool_index = pool_index;
  A.px = pool_x; A.py = pool_y; A.ph = pool_heading; A.pv = pool_speed; A.pvx = pool_vx; A.pvy = pool_vy;
  A.goal_last_pose = c->goal_last_pose; A.goal_noact_count = c->goal_noact_count;
  A.wheel_f = c->wheel_f; A.wheel_r = c->wheel_r; A.pool_wf = c->reset_pool_wf; A.pool_wr = c->reset_pool_wr;
  A.last_accel = c->ctrl_last_accel; A.type_id = c->type_id; A.table = c->d_table; A.n_types = c->n_types;
  A.N = c->N; A.M = c->M; A.n_pool = n_pool;
  const long long total = (long long)c->N * c->M;
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)c->sm_count * 8);
  t2d_reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

int t2d_lidar_scan(t2d_ctx* c, int n_beams, float max_range, const double* beam_cos_sin, float* scan, void* stream) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!c->x) return fail(T2D_E_STATE, "state not bound: call t2d_bind_state first");
  if (!c->d_table || c->n_types == 0) return fail(T2D_E_STATE, "type table not set: call t2d_set_type_table first");
  if (n_beams <= 0 || !(max_range > 0.0f) || !beam_cos_sin || !scan) return fail(T2D_E_INVALID, "t2d_lidar_scan: bad argument");
  CUDA_TRY(cudaSetDevice(c->device));
  LidarArgs A{};
  A.x = c->x; A.y = c->y; A.h = c->h; A.type_id = c->type_id; A.table = c->d_table; A.n_types = c->n_types;
  A.map_blob = c->d_map; A.tile_off = c->d_tile_off; A.tile_id = c->n_tiles > 1 ? c->tile_id : nullptr;
  A.beam_cs = beam_cos_sin; A.scan = scan;
  A.N = c->N; A.M = c->M; A.n_beams = n_beams; A.range = (double)max_range;
  const int grid = (c->N + LIDAR_WARPS - 1) / LIDAR_WARPS;
  t2d_lidar_kernel<<<grid, LIDAR_WARPS * 32, 0, (cudaStream_t)stream>>>(A);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

int t2d_set_controllers(t2d_ctx* c, const t2d_controller_params* table, int n_rows, const uint8_t* ctrl_id,
                        const int16_t* lead_index, const int16_t* path_id, float* last_accel) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  CUDA_TRY(cudaSetDevice(c->device));
  if (!table) {
    if (c->d_ctab) cudaFree(c->d_ctab);
    c->d_ctab = nullptr; c->n_ctrl = 0; c->ctrl_id = nullptr; c->ctrl_lead = nullptr; c->ctrl_path = nullptr;
    c->ctrl_last_accel = nullptr;
    return T2D_OK;
  }
  if (n_rows <= 0 || n_rows > T2D_MAX_CONTROLLERS) return fail(T2D_E_INVALID, "n_rows must be in 1..T2D_MAX_CONTROLLERS");
  if (!ctrl_id || !last_accel) return fail(T2D_E_INVALID, "t2d_set_controllers: ctrl_id / last_accel is NULL");
  for (int i = 0; i < n_rows; ++i) {
    const t2d_controller_params& p = table[i];
    if (p.kind < T2D_CTRL_EXTERNAL || p.kind > T2D_CTRL_PURE_PURSUIT) return fail(T2D_E_INVALID, "unknown controller kind");
    if (p.kind == T2D_CTRL_PURE_PURSUIT && !(p.min_pre_aiming_distance > 0.0f))
      return fail(T2D_E_INVALID, "min_pre_aiming_distance must be positive");   // pure_pursuit_controller.py:30-31
    if (p.kind >= T2D_CTRL_CRUISE && p.target_speed < 0.0f)
      return fail(T2D_E_INVALID, "target_speed must be non-negative");          // acceleration_controller.py:48-49
  }
  if (c->d_ctab) { cudaFree(c->d_ctab); c->d_ctab = nullptr; }
  CUDA_TRY(cudaMalloc(&c->d_ctab, sizeof(t2d_controller_params) * n_rows));
  CUDA_TRY(cudaMemcpy(c->d_ctab, table, sizeof(t2d_controller_params) * n_rows, cudaMemcpyHostToDevice));
  c->n_ctrl = n_rows; c->ctrl_id = ctrl_id; c->ctrl_lead = lead_index; c->ctrl_path = path_id; c->ctrl_last_accel = last_accel;
  return T2D_OK;
}

int t2d_set_paths(t2d_ctx* c, const float* xy, const int32_t* offsets, int n_paths) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  CUDA_TRY(cudaSetDevice(c->device));
  if (c->d_path_v) { cudaFree(c->d_path_v); c->d_path_v = nullptr; }
  if (c->d_path_off) { cudaFree(c->d_path_off); c->d_path_off = nullptr; }
  c->n_paths = 0;
  if (n_paths == 0 || !xy) return T2D_OK;
  if (n_paths < 0 || !offsets) return fail(T2D_E_INVALID, "t2d_set_paths: bad argument");
  if (offsets[0] != 0) return fail(T2D_E_INVALID, "offsets[0] must be 0");
  for (int p = 0; p < n_paths; ++p)
    if (offsets[p + 1] - offsets[p] < 2) return fail(T2D_E_INVALID, "a path needs at least 2 vertices");
  const int V = offsets[n_paths];
  std::vector<PathVertex> pv((size_t)V);
  for (int p = 0; p < n_paths; ++p) {
    double acc = 0.0;   // the running arc length of LineString.interpolate's walk, in float64
    for (int i = offsets[p]; i < offsets[p + 1]; ++i) {
      pv[i].x = xy[2 * i]; pv[i].y = xy[2 * i + 1];
      pv[i].cum = acc;
      pv[i].len = 0.0;
      if (i + 1 < offsets[p + 1]) {
        pv[i].len = hypot((double)xy[2 * i + 2] - (double)xy[2 * i], (double)xy[2 * i + 3] - (double)xy[2 * i + 1]);
        acc += pv[i].len;
      }
    }
  }
  CUDA_TRY(cudaMalloc(&c->d_path_v, sizeof(PathVertex) * (size_t)V));
  CUDA_TRY(cudaMemcpy(c->d_path_v, pv.data(), sizeof(PathVertex) * (size_t)V, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMalloc(&c->d_path_off, sizeof(int) * (size_t)(n_paths + 1)));
  CUDA_TRY(cudaMemcpy(c->d_path_off, offsets, sizeof(int) * (size_t)(n_paths + 1), cudaMemcpyHostToDevice));
  c->n_paths = n_paths;
  return T2D_OK;
}

int t2d_control(t2d_ctx* c, float* action, void* stream) {
  if (!c) return fail(T2D_E_INVALID, "ctx is NULL");
  if (!c->x) return fail(T2D_E_STATE, "state not bound: call t2d_bind_state first");
  if (!c->d_table || c->n_types == 0) return fail(T2D_E_STATE, "type table not set: call t2d_set_type_table first");
  if (!c->d_ctab) return fail(T2D_E_STATE, "controllers not set: call t2d_set_controllers first");
  if (!action) return fail(T2D_E_INVALID, "action is NULL");
  if (reinterpret_cast<uintptr_t>(action) % 8 != 0) return fail(T2D_E_INVALID, "action must be 8-byte aligned");
  CUDA_TRY(cudaSetDevice(c->device));
  CtrlArgs A{};
  A.x = c->x; A.y = c->y; A.h = c->h; A.v = c->v; A.type_id = c->type_id; A.table = c->d_table; A.n_types = c->n_types;
  A.ctab = c->d_ctab; A.n_ctrl = c->n_ctrl; A.ctrl_id = c->ctrl_id; A.lead = c->ctrl_lead; A.path_id = c->ctrl_path;
  A.path_v = c->d_path_v; A.path_off = c->d_path_off; A.n_paths = c->n_paths;
  A.last_accel = c->ctrl_last_accel; A.action = action; A.ego_action = c->ego_action;
  A.N = c->N; A.M = c->M; A.steer_first = (c->cfg.flags & T2D_CFG_STEER_FIRST) ? 1 : 0;
  const int warps_per_cta = 4;
  const int grid = std::max(1, std::min((c->N + warps_per_cta - 1) / warps_per_cta, c->sm_count * 16));
  t2d_control_kernel<<<grid, warps_per_cta * 32, 0, (cudaStream_t)stream>>>(A);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

int t2d_exchange_create(t2d_exchange** out, int device, int world, int rank, int n_local, int slots, void* ipc_handle_out) {
  if (!out || !ipc_handle_out) return fail(T2D_E_INVALID, "out / ipc_handle_out is NULL");
  *out = nullptr;
  if (world < 1 || world > T2D_MAX_RANKS || rank < 0 || rank >= world) return fail(T2D_E_INVALID, "bad world / rank");
  if (n_local <= 0 || slots < 2 || slots > 64) return fail(T2D_E_INVALID, "n_local must be > 0 and slots in 2..64");
  static_assert(sizeof(cudaIpcMemHandle_t) == T2D_IPC_HANDLE_BYTES, "IPC handle size");
  CUDA_TRY(cudaSetDevice(device));
  t2d_exchange* x = new t2d_exchange();
  x->device = device; x->world = world; x->rank = rank; x->n_real = n_local; x->n_local = (n_local + 15) & ~15; x->slots = slots;
  x->threads = std::min(256, 32 * world);                 // one warp per peer
  if (const char* e = getenv("T2D_EXCHANGE_THREADS")) {   // experiments: a smaller CTA finds a home on a busy SM sooner
    const int v = atoi(e);
    if (v >= 32 && v <= 512 && v % 32 == 0 && v >= world) x->threads = v;
  }
  if (const char* e = getenv("T2D_EXCHANGE_TIMEOUT_MS")) {
    const double ms = atof(e);
    if (ms > 0.0) x->timeout_cycles = (long long)(ms * 2.0e6);   // ~2 GHz SM clock
  }
  x->bytes = x->flag_off() + (T2D_MAX_RANKS + 4) * sizeof(unsigned);
  cudaError_t e = cudaMalloc(&x->base, x->bytes);
  if (e == cudaSuccess) e = cudaMemset(x->base, 0, x->bytes);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, x->base);
  if (e != cudaSuccess) {
    if (x->base) cudaFree(x->base);
    delete x;
    return fail(T2D_E_CUDA, std::string("t2d_exchange_create: ") + cudaGetErrorString(e));
  }
  memcpy(ipc_handle_out, &h, sizeof(h));
  CUDA_TRY(cudaDeviceSynchronize());
  g_exchanges_alive.fetch_add(1);
  *out = x;
  return T2D_OK;
}

int t2d_exchange_connect(t2d_exchange* x, const void* handles) {
  if (!x || !handles) return fail(T2D_E_INVALID, "exchange / handles is NULL");
  CUDA_TRY(cudaSetDevice(x->device));
  for (int p = 0; p < x->world; ++p) {
    if (p == x->rank) { x->peer[p] = x->base; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const unsigned char*>(handles) + (size_t)p * sizeof(h), sizeof(h));
    void* ptr = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {   // do not leak the mappings opened so far
      for (int q = 0; q < p; ++q)
        if (q != x->rank && x->peer[q]) { cudaIpcCloseMemHandle(x->peer[q]); x->peer[q] = nullptr; }
      return fail(T2D_E_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    }
    x->peer[p] = static_cast<unsigned char*>(ptr);
  }
  x->connected = true;
  return T2D_OK;
}

int t2d_exchange_allgather_lagged(t2d_exchange* x, const uint8_t* done_local, uint8_t* dst, int lag, void* stream) {
  if (!x || !done_local || !dst) return fail(T2D_E_INVALID, "exchange / done_local / dst is NULL");
  if (!x->connected) return fail(T2D_E_STATE, "exchange not connected: call t2d_exchange_connect first");
  if (lag < 0 || 2 * lag + 2 > x->slots) return fail(T2D_E_INVALID, "lag needs a ring of at least 2 * lag + 2 slots");
  CUDA_TRY(cudaSetDevice(x->device));
  AllGatherArgs A{};
  for (int p = 0; p < x->world; ++p) A.peer[p] = x->peer[p];
  A.base = x->base; A.local = done_local; A.dst = dst;
  A.world = x->world; A.rank = x->rank; A.n_local = x->n_local; A.n_real = x->n_real; A.slots = x->slots;
  A.lag = lag; A.timeout = x->timeout_cycles;
  t2d_exchange_allgather_kernel<<<1, x->threads, 0, (cudaStream_t)stream>>>(A);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

int t2d_exchange_allgather(t2d_exchange* x, const uint8_t* done_local, uint8_t* dst, void* stream) {
  return t2d_exchange_allgather_lagged(x, done_local, dst, 0, stream);
}

int t2d_exchange_status(t2d_exchange* x, uint32_t* steps, uint32_t* timed_out) {
  if (!x) return fail(T2D_E_INVALID, "exchange is NULL");
  CUDA_TRY(cudaSetDevice(x->device));
  unsigned w[4];
  CUDA_TRY(cudaMemcpy(w, x->word(0), sizeof(w), cudaMemcpyDeviceToHost));
  if (steps) *steps = w[0];
  if (timed_out) *timed_out = w[3];
  return T2D_OK;
}

int t2d_exchange_destroy(t2d_exchange* x) {
  if (!x) return T2D_OK;
  cudaSetDevice(x->device);
  for (int p = 0; p < x->world; ++p)
    if (x->connected && p != x->rank && x->peer[p]) cudaIpcCloseMemHandle(x->peer[p]);
  if (x->base) cudaFree(x->base);
  g_exchanges_alive.fetch_sub(1);
  delete x;
  return T2D_OK;
}

int t2d_physics_step(int device, const t2d_type_params* params, int interval_ms, int delta_t_ms, int n, float* x, float* y,
                     float* heading, float* speed, float* vx, float* vy, float* omega_front, float* omega_rear,
                     const float* action, float* applied, void* stream) {
  if (!params) return fail(T2D_E_INVALID, "params is NULL");
  if (n < 0) return fail(T2D_E_INVALID, "n must be >= 0");
  if (n == 0) return T2D_OK;
  if (!x || !y || !heading || !speed || !vx || !vy || !action) return fail(T2D_E_INVALID, "t2d_physics_step: NULL array");
  if (interval_ms <= 0 || delta_t_ms <= 0) return fail(T2D_E_INVALID, "interval_ms and delta_t_ms must be > 0");
  if (params->model < 0 || params->model > T2D_MODEL_DRIFT) return fail(T2D_E_INVALID, "unknown model id");
  if (params->model == T2D_MODEL_DRIFT && !(omega_front && omega_rear))
    return fail(T2D_E_INVALID, "t2d_physics_step: SingleTrackDrift needs the wheel-speed arrays");
  CUDA_TRY(cudaSetDevice(device));
  PhysArgs A{};
  A.wheel_f = omega_front; A.wheel_r = omega_rear;
  {
    AbiParams a;
    memcpy(&a, params, sizeof(AbiParams));
    A.p = derive_params(a);
  }
  A.x = x; A.y = y; A.h = heading; A.v = speed; A.vx = vx; A.vy = vy; A.action = action; A.applied = applied;
  A.n = n;
  const int delta_t = std::min(delta_t_ms, interval_ms);
  A.n_steps = interval_ms / delta_t;
  A.dt = (float)((double)delta_t / 1000.0);
  A.dt_rem = (float)((double)(interval_ms % delta_t) / 1000.0);
  A.dt_d = (double)delta_t / 1000.0;
  A.dt_rem_d = (double)(interval_ms % delta_t) / 1000.0;
  A.interval_d = (double)interval_ms / 1000.0;
  const int grid = std::min((n + 255) / 256, 148 * 8);
  t2d_physics_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  return T2D_OK;
}

}  // extern "C"
