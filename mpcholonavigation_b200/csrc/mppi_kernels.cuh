// mppi_kernels.cuh -- the sm_100a kernels of the MPPI hot path.
//
//  K1 noise_philox_kernel          NoiseGenerator::generateNoisedControls   (noise_generator.cpp:107-122)
//  K2 rollout_score_kernel         setNoisedControls + updateStateVelocities + predict + integrateStateVelocities
//                                  + every critic that does not need the furthest path point
//                                  (noise_generator.cpp:65-74, optimizer.cpp:251-273,313-343, motion_models.hpp:53-66,
//                                   src/critics/{constraint,cost,goal,goal_angle,obstacles,prefer_forward,twirling,
//                                   velocity_deadband}_critic.cpp, utils.hpp:292-319)
//  K3 path_softmax_update_kernel   PathFollow / PathAlign / PathAlignLegacy / PathAngle critics, cost totals in list
//                                  order with the fail_flag short-circuit, gamma term, softmax weights and the
//                                  weighted control update, clip  (critic_manager.cpp:67-76, path_*_critic.cpp,
//                                  optimizer.cpp:362-394,237-249)
//  K4 merge_finalize_kernel        parallel merge of the softmax partials (large batches; cross-rank when sharded)
//  KF tile_fused_kernel            small batches, one rank: K2's body, both grid-wide exchanges (as packets), the path critics,
//                                  the update, the merge and the evalControl tail in ONE cooperative launch; zero-copy upload
//                                  in, result packets out (the default 1000 x 56 path)
//     *_batch_kernel (stream)     K2 / K3a / K3c / K4 of the stream layout with the robot as the last grid dimension
//                                  (and K1's regenerate_noises redraw, noise_philox_batch_kernel)
//
// Work shape of K2: one CTA owns a tile of 32 trajectories (lane == trajectory) and S warps split the
// horizon into S contiguous segments.  The tile lives in shared memory time-major, [T][33] floats per
// plane, which is bank-conflict free both for the coalesced row-major global load (lane == t) and for the
// per-trajectory accesses (lane == trajectory).  The three cumulative sums (yaw, x, y) are evaluated
// SEQUENTIALLY in t by one lane per trajectory with non-contractable fp32 adds: this is the reference's
// summation order, and it is what makes the costmap cell indices bit-exact against the CPU oracle.
// Everything else (sincos, costmap gathers, critic terms) is evaluated in parallel over (trajectory, t).
#pragma once
#include <cuda.h>
#include <type_traits>

#include "mppi_device.cuh"

namespace mppi
{

// Programmatic dependent launch (griddepcontrol): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization
// may start while its predecessor on the stream is still draining; it runs the part of its prologue that does not read the
// predecessor's results (record and path tables into shared memory, mbarrier set-up, the first TMA loads of the static noise
// planes) and then waits.  pdl_wait() returns at once in a kernel that was launched the ordinary way.
__device__ __forceinline__ void pdl_launch_dependents() {asm volatile ("griddepcontrol.launch_dependents;" ::: "memory");}
__device__ __forceinline__ void pdl_wait() {asm volatile ("griddepcontrol.wait;" ::: "memory");}

// shared-window addressing by 32-bit address (the tables a kernel reads with data-dependent indices: generic pointers make
// the compiler rebuild the window base at every access)
__device__ __forceinline__ unsigned smem_addr(const void * p) {return static_cast<unsigned>(__cvta_generic_to_shared(p));}
__device__ __forceinline__ float lds_f32(unsigned a) {float v; asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v;}
__device__ __forceinline__ unsigned lds_u8(unsigned a) {unsigned v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v;}

struct DevBuffers
{
  const float * in_a;   // mode 0: noise vx | mode 1,2: state vx      [B][T]
  const float * in_b;   //         noise vy |            state vy
  const float * in_c;   //         noise wz |            state wz
  const float * in_x;   // mode 2: trajectories x, y, yaw             [B][T]
  const float * in_y;
  const float * in_yaw;
  float * cs;           // control sequence [3][T]: vx, vy, wz
  float * crit_rows;    // [n_critics + 3][B]
  float * samples_x;    // [K][B]
  float * samples_y;
  float * samples_yaw;
  float * end_xy;       // [2][B]
  float * spill_x;      // [T][B]
  float * spill_y;
  float * spill_yaw;
  int * spill_cells;    // [T][B]
  float * vis_xy;       // [2][ceil(T / vis_t_step)][ceil(B / vis_b_step)] sub-sampled x, y for the TrajectoryVisualizer
  float * costs;        // [B]
  float * partials;     // [blocks][3T + 2]
  float * rank_partial; // [3T + 2] (+ fail flag / furthest packed after it for the exchange)
  float * out;          // [3T + 4]: new control sequence, fail flag, furthest (as bit patterns)
  DevState * st;
  PeerComm peer;        // sharded over peer memory when peer.nranks > 1
  // fused small-batch kernel: the exchanges between the tiles of one launch travel as self-validating packets
  // {value, tag of the launch} (the protocol of the peer exchange above, inside one GPU)
  uint2 * pk_up;        // [G]            per tile: "my slice of the upload is in device memory"
  uint2 * pk_x1;        // [G]            per tile: furthest-point candidate | survivor flags << 16
  uint2 * pk_rec;       // [G][3T + 2]    per tile: softmax record (m, s, W[3T])
  uint2 * pk_out;       // [3T]           evalControl tail: the new sequence on its way from the owner tiles to tile 0
  unsigned * epoch;     // completed fused launches of this handle; the tag of the running launch is *epoch + 1
  unsigned * host_err;  // pinned host word (behind the result packets): a bounded poll gave up inside this handle's kernels
};

// A bounded poll timed out: sticky flag in device memory and, for the cycles whose result leaves as packets (no D2H of the
// state), in pinned host memory too.  The system-scope fence orders the host word before every packet this block sends
// afterwards, and the result packets are only sent once every tile's packets have arrived: the host reads the word after
// the last result packet and cannot miss it.
__device__ __forceinline__ void raise_comm_error(const DevBuffers & bufs)
{
  bufs.st->comm_error = 1u;
  if (bufs.host_err) {
    *reinterpret_cast<volatile unsigned *>(bufs.host_err) = 1u;
    __threadfence_system();
  }
}

// accumulator slots of the per-segment partials
enum Acc
{
  A_CON = 0, A_FWD, A_TWIRL, A_DB, A_GOAL, A_GANG, A_GVX, A_GVY, A_GWZ, A_COST_REP, A_COST_HIT, A_OB_TRAJ, A_OB_REP,
  A_OB_HIT, A_COUNT
};

// shared memory of K2: hot params + control sequence + initial velocities + tile planes + partials + argmin scratch.
// Rollout modes keep 4 planes (x and y are built IN PLACE over the vx / vy control planes once the velocity
// critics have consumed them); the score mode (caller-provided trajectories) needs x and y beside the state: 6.
__host__ __device__ inline int rollout_planes(int mode) {return mode == 2 ? 6 : 4;}
__host__ __device__ inline size_t rollout_smem_floats(int T, int S, int planes)
{
  return static_cast<size_t>(kHotFloats) + 3 * T + 3 * kTile + static_cast<size_t>(planes) * T * kPad +
         static_cast<size_t>(S) * A_COUNT * kTile + 2 * static_cast<size_t>(S) * kTile;
}
__host__ __device__ inline size_t rollout_smem_bytes(int T, int S, int mode)
{
  return sizeof(float) * rollout_smem_floats(T, S, rollout_planes(mode));
}

// The fused small-batch kernel (tile_fused_kernel, below) keeps going where K2 stops: what K2 leaves in shared memory
// and registers is handed over in this record instead of through global memory.
struct FusedShared
{
  float * rows;       // [kMaxCritics + kGammaRows][32] per-critic contributions of this tile + the three gamma sums
  float * term;       // [4][32] path critic terms: follow, align, legacy, angle
  float * w;          // [32] softmax weights of the tile
  float * stat;       // [8]  m, sum of weights
  float * D, * px, * py;        // [N] arc-length prefix and points of the path
  uint8_t * valid, * flags;     // [n16]
  uint16_t * follow;            // [N]
  float * e;          // [G] rescale factors of the merge
  float * red;        // [32] block reductions
  float * ap;         // [8][2][32] PathAlign: per-warp partial (sum, count) of every trajectory
  float * ad;         // [n_s][32]  PathAlign: segment length -> integrated distance of every sampled pose; behind it
                      // [n_s][32]  int: lower bound | candidate << 16 -> chosen path point
};
// n_s: sampled poses of PathAlign (0 when the critic is not in the list)
__host__ __device__ inline size_t fused_extra_floats(int N, int G, int n_s)
{
  const int n16 = ((N + 15) / 16) * 16;
  return static_cast<size_t>(kMaxCritics + kGammaRows) * kTile + 4 * kTile + kTile + 8 + 3 * static_cast<size_t>(n16) +
         n16 / 2 /* valid + flags bytes */ + n16 / 2 /* follow uint16 */ + static_cast<size_t>(((G + 31) / 32) * 32) + 32 +
         8 * 2 * kTile + 2 * static_cast<size_t>(n_s) * kTile;
}
__host__ __device__ inline size_t fused_smem_bytes(int T, int S, int N, int G, int n_s)
{
  return sizeof(float) * (rollout_smem_floats(T, S, 6) + fused_extra_floats(N, G, n_s));
}
__device__ __forceinline__ FusedShared fused_carve(float * base, int N, int G)
{
  const int n16 = ((N + 15) / 16) * 16;
  FusedShared f;
  f.rows = base;
  f.term = f.rows + (kMaxCritics + kGammaRows) * kTile;
  f.w = f.term + 4 * kTile;
  f.stat = f.w + kTile;
  f.D = f.stat + 8;
  f.px = f.D + n16;
  f.py = f.px + n16;
  f.valid = reinterpret_cast<uint8_t *>(f.py + n16);
  f.flags = f.valid + n16;
  f.follow = reinterpret_cast<uint16_t *>(f.flags + n16);
  f.e = reinterpret_cast<float *>(f.follow + n16);
  f.red = f.e + ((G + 31) / 32) * 32;
  f.ap = f.red + 32;
  f.ad = f.ap + 8 * 2 * kTile;
  return f;
}
// what the K2 body hands to the fused tail
struct FusedCtx
{
  FusedShared fs;
  const float * s_hot, * s_cs;
  const float * s_cvx, * s_cvy, * s_cwz, * s_yaw, * s_x, * s_y;   // time-major tile planes [T][33]
  int n_cap, iteration;   // n_cap: path capacity the shared-memory carve-up was sized for (>= the record's N)
  int tile, ntiles;       // this block's tile of the problem and the number of tiles (blockIdx.x / gridDim.x)
  unsigned tag;           // tag of this launch's packets
  // zero-copy upload: the cycle's record + costmap sit in pinned host memory (up_host, up_vecs 16-byte vectors, laid
  // out like the device buffer that starts at the record); every tile reads the hot part of the record straight from
  // there and copies one slice of the whole into device memory, where the cold parts and the costmap are read once all
  // tiles have signalled (before the first costmap access).  nullptr: the buffers are already resident.
  const uint4 * up_host;
  int up_vecs;
};

// ---------------------------------------------------------------------------------------------------
// K1: Philox4x32-10 + Box-Muller.  One thread = one trajectory x one quad of time steps x 3 planes;
// counter = (t/4, plane, global trajectory, stream), key = seed: shards of a sharded batch tile exactly.
// Stores are float4 (coalesced along t) when T % 4 == 0.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4])
{
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;}
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0;
    const uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float & z0, float & z1)
{
  const float u1 = static_cast<float>((a >> 8) + 1u) * 5.9604644775390625e-08f;   // (0,1]
  const float u2 = static_cast<float>(b >> 8) * 5.9604644775390625e-08f;          // [0,1)
  const float r = __fsqrt_rn(__fmul_rn(-2.0f, logf(u1)));
  float s, c;
  mppi_det_sincosf(__fmul_rn(6.283185307179586f, u2), &s, &c);
  z0 = __fmul_rn(r, c);
  z1 = __fmul_rn(r, s);
}

// one noise set (three planes) of one handle, grid-stride over blockIdx.x; shared by the single-handle and group kernels
// so that both draw the same bits for the same (seed, stream)
__device__ __forceinline__ void noise_philox_body(
  float * __restrict__ nvx, float * __restrict__ nvy, float * __restrict__ nwz, int B, int T, float sx, float sy, float sw,
  int holonomic, uint64_t seed, uint64_t stream, uint64_t shard_offset, int time_major)
{
  const int quads = (T + 3) >> 2;
  const long long total = static_cast<long long>(B) * quads;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
    i += static_cast<long long>(gridDim.x) * blockDim.x)
  {
    // row-major [B][T]: consecutive threads walk t (float4 stores); time-major [T][B]: consecutive threads walk b
    const int b = time_major ? static_cast<int>(i % B) : static_cast<int>(i / quads);
    const int q = time_major ? static_cast<int>(i / B) : static_cast<int>(i - static_cast<long long>(b) * quads);
    const uint32_t gb = static_cast<uint32_t>(static_cast<uint64_t>(b) + shard_offset);
#pragma unroll
    for (int plane = 0; plane < 3; ++plane) {
      float * dst = plane == 0 ? nvx : (plane == 1 ? nvy : nwz);
      const float sd = plane == 0 ? sx : (plane == 1 ? sy : sw);
      float z[4] = {0.f, 0.f, 0.f, 0.f};
      if (plane != 1 || holonomic) {
        uint32_t r[4];
        philox4x32_10(static_cast<uint32_t>(q), static_cast<uint32_t>(plane), gb, static_cast<uint32_t>(stream),
          static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), r);
        box_muller(r[0], r[1], z[0], z[1]);
        box_muller(r[2], r[3], z[2], z[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {z[j] = __fmul_rn(z[j], sd);}
      }
      if (time_major) {
        for (int j = 0; j < 4 && 4 * q + j < T; ++j) {dst[static_cast<size_t>(4 * q + j) * B + b] = z[j];}
      } else {
        float * row = dst + static_cast<size_t>(b) * T + 4 * q;
        if ((T & 3) == 0) {
          *reinterpret_cast<float4 *>(row) = make_float4(z[0], z[1], z[2], z[3]);
        } else {
          for (int j = 0; j < 4 && 4 * q + j < T; ++j) {row[j] = z[j];}
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) noise_philox_kernel(
  float * __restrict__ nvx, float * __restrict__ nvy, float * __restrict__ nwz, int B, int T, float sx, float sy, float sw,
  int holonomic, uint64_t seed, uint64_t stream, uint64_t shard_offset, int time_major, const unsigned long long * __restrict__ d_epoch)
{
  // regenerate_noises: the Philox stream index lives in device memory so that a captured graph draws a new set per replay
  if (d_epoch) {stream = *d_epoch;}
  noise_philox_body(nvx, nvy, nwz, B, T, sx, sy, sw, holonomic, seed, stream, shard_offset, time_major);
}

// regenerate_noises members of a robot group (unsharded, stream layout): what launch_regenerate passes for one handle
struct __align__(16) NoiseJob
{
  float * noise[3];
  unsigned long long * epoch;   // the member's Philox stream index of the next draw
  uint64_t seed;
  int B, T;
  float sx, sy, sw;
  int holonomic;
};
static_assert(sizeof(NoiseJob) % 16 == 0, "the noise table is an array of 16-byte aligned records");

// the redraw of every listed member in one launch (member = blockIdx.y), bit-equal to noise_philox_kernel per member
__global__ void __launch_bounds__(256) noise_philox_batch_kernel(const NoiseJob * __restrict__ jobs)
{
  const NoiseJob & j = jobs[blockIdx.y];
  noise_philox_body(j.noise[0], j.noise[1], j.noise[2], j.B, j.T, j.sx, j.sy, j.sw, j.holonomic, j.seed, *j.epoch, 0, 1);
}

// Compile-time feature sets of the K2 kernels.  An EXACT instance (kExact) is straight-line code for one set of active
// features (no per-cycle flag tests, no dead critic code: smaller, fewer registers, fewer instruction-cache misses);
// the generic instance (SF_ALL, !kExact) tests the per-cycle flags of the record at run time.  The host picks the exact
// instance when the cycle's record asks for precisely that set (launch_rollout), else the generic one.
enum StreamFeature : unsigned
{
  SF_HOL = 1u,          // holonomic (Omni): vy terms
  SF_ACKER = 2u,        // Ackermann term of the Constraint critic
  SF_CON = 4u,          // ConstraintCritic
  SF_FWD = 8u,          // PreferForwardCritic
  SF_TWIRL = 16u,       // TwirlingCritic
  SF_DB = 32u,          // VelocityDeadbandCritic
  SF_GOAL = 64u,        // GoalCritic
  SF_GANG = 128u,       // GoalAngleCritic
  SF_COST = 256u,       // CostCritic
  SF_OBST = 512u,       // ObstaclesCritic
  SF_FOOTPRINT = 1024u, // footprint-cost mode of either costmap critic
  SF_SPILL = 2048u,     // trajectories / cell indices written out
  SF_ALL = 4095u
};
#define MPPI_SF(bit, flag) (((F & (bit)) != 0) && (kExact || (flag)))

__global__ void advance_epoch_kernel(unsigned long long * d_epoch) {*d_epoch += 1ull;}

// the same for n members of a robot group, behind their noise_philox_batch_kernel
__global__ void advance_epoch_batch_kernel(const NoiseJob * __restrict__ jobs, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {*jobs[i].epoch += 1ull;}
}

// ---------------------------------------------------------------------------------------------------
// K2
// ---------------------------------------------------------------------------------------------------
#ifndef MPPI_K2_MIN_BLOCKS
#define MPPI_K2_MIN_BLOCKS 3
#endif
#ifndef MPPI_TILE_CHUNK
#define MPPI_TILE_CHUNK 1
#endif
constexpr int kTileChunk = MPPI_TILE_CHUNK;   // steps whose independent work is issued together inside a segment
template<unsigned F, bool kExact, int kMode, bool kFused>
__device__ __forceinline__ void rollout_tile_body(
  const DevParams * P, const uint8_t * cm, const DevBuffers & bufs, const int B, const int T, FusedCtx * fx)
{
  // the fused kernels' tiles WRITE the device copy of [record | costmap] in this very launch (zero-copy upload): no
  // non-coherent loads from either there (ld_ro); the two-kernel instances keep ld.global.nc
  constexpr bool kNc = !kFused;
  constexpr int mode = kMode;   // 0 rollout from noise, 1 injected state (integrate), 2 injected state + trajectories
  static_assert(!kFused || kMode == 0, "the fused kernel only exists for the rollout-from-noise mode");
  // B, T and mode also live in the record, but as launch arguments they cost no memory round trip: the noise rows,
  // the control sequence and the record are all requested at once when the kernel starts
  extern __shared__ float smem[];
  const int S = blockDim.y;
  const int lane = threadIdx.x, seg = threadIdx.y;
  const int tid = seg * kTile + lane;
  const int tile = kFused ? fx->tile : static_cast<int>(blockIdx.x);
  const int ntiles = kFused ? fx->ntiles : static_cast<int>(gridDim.x);
  const int nthreads = S * kTile;

  float * s_hot = smem;
  const DevParams & p = *reinterpret_cast<const DevParams *>(s_hot);
  const int tplane = T * kPad;
  float * s_cs = s_hot + kHotFloats;             // [3][T]
  float * s_v0 = s_cs + 3 * T;                   // [3][32] initial velocities per trajectory
  float * s_cvx = s_v0 + 3 * kTile;              // controls vx  -> (rollout modes) x
  float * s_cvy = s_cvx + tplane;                // controls vy  -> (rollout modes) y
  float * s_cwz = s_cvy + tplane;                // controls wz
  float * s_yaw = s_cwz + tplane;
  constexpr bool kSixPlanes = mode == 2 || kFused;   // x and y beside the controls (the fused tail re-reads the controls)
  float * s_x = kSixPlanes ? s_yaw + tplane : s_cvx;
  float * s_y = kSixPlanes ? s_x + tplane : s_cvy;
  float * s_acc = s_yaw + tplane * (kSixPlanes ? 3 : 1);   // [S][A_COUNT][32]
  float * s_amin_d = s_acc + S * A_COUNT * kTile;         // [S][32]
  int * s_amin_j = reinterpret_cast<int *>(s_amin_d + S * kTile);
  FusedShared fs = {};
  if (kFused) {
    fs = fused_carve(reinterpret_cast<float *>(s_amin_j + S * kTile), fx->n_cap, ntiles);
    fx->fs = fs;
    fx->s_hot = s_hot; fx->s_cs = s_cs; fx->s_cvx = s_cvx; fx->s_cvy = s_cvy; fx->s_cwz = s_cwz; fx->s_yaw = s_yaw;
    fx->s_x = s_x; fx->s_y = s_y;
    if (tid == 0) {reinterpret_cast<unsigned *>(fs.stat)[7] = 0u;}   // exchange-1 word of this tile, gathered in P6
  }

  const int b0 = tile * kTile;
  const int b = b0 + lane;
  const bool live = b < B;

  MPPI_TRACE_AT(0);
  // ---- P1: stage the tile.  Everything this block needs from global memory is REQUESTED before anything is consumed
  //      (the first touch of global memory costs ~1 us even on an L2 hit, so dependent waves are what to avoid): the hot
  //      part of the record and the control sequence go to registers first, then the noise rows, then all of it is
  //      stored to shared memory.
  const bool zero_copy = kFused && fx->up_host != nullptr;
  const float4 * hot_src = zero_copy ? reinterpret_cast<const float4 *>(fx->up_host) : reinterpret_cast<const float4 *>(P);
  float4 hot_v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (tid < kHotBytes / 16) {hot_v = __ldg(hot_src + tid);}
  // zero-copy upload: this tile's slice of [record | costmap], two vectors per thread in flight, the rest (large
  // costmaps) in a plain loop behind the staging
  // (the copy is the business of the warps that have no scan to do: requested now, stored and fenced while warp 0 walks
  //  the yaw scan, so that neither the PCIe latency nor the fence sits on the path of a barrier)
  uint4 up_v[2] = {make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u)};
  int up_begin = 0, up_end = 0;
  const int up_tid = S > 1 ? tid - kTile : tid, up_n = S > 1 ? nthreads - kTile : nthreads;   // warp 0 sits out when it can
  if (kFused) {
    if (zero_copy && up_tid >= 0) {
      const int per = (fx->up_vecs + ntiles - 1) / ntiles;
      up_begin = min(fx->up_vecs, tile * per);
      up_end = min(fx->up_vecs, up_begin + per);
      if (up_begin + up_tid < up_end) {up_v[0] = __ldg(fx->up_host + up_begin + up_tid);}
      if (up_begin + up_n + up_tid < up_end) {up_v[1] = __ldg(fx->up_host + up_begin + up_n + up_tid);}
    }
  }
  float cs_v[2] = {0.0f, 0.0f};
  if (tid < 3 * T) {cs_v[0] = bufs.cs[tid];}
  if (tid + nthreads < 3 * T) {cs_v[1] = bufs.cs[tid + nthreads];}
  if (mode == 0) {
    // Warp `seg` owns rows seg, seg+S, ...; lane walks t (coalesced 128 B rows).  A batch = kCols 32-step columns x 4
    // rows (fused: 2 x 4 covers the tile in one wave for T <= 64 with 8 warps; the two-kernel instances run at 3 blocks
    // per SM and keep fewer loads in flight).  The control sequence of the batch's columns rides in the same wave, so
    // setNoisedControls (noise_generator.cpp:71-73), c = control_sequence + noise, happens on the way into the tile.
    constexpr int kCols = kFused ? 2 : 1, kRows = 4;
    const int ncol = (T + 31) >> 5;
    const int nri = (kTile - seg + S - 1) / S;
    for (int ri0 = 0; ri0 < nri; ri0 += kRows) {
      for (int ci0 = 0; ci0 < ncol; ci0 += kCols) {
        float ca[kCols], cb[kCols], cc[kCols];
        float va[kCols][kRows], vb[kCols][kRows], vc[kCols][kRows];
        int oo[kCols][kRows];
#pragma unroll
        for (int c = 0; c < kCols; ++c) {
          const int t = ((ci0 + c) << 5) + lane;
          const bool okc = ci0 + c < ncol && t < T;
          ca[c] = cb[c] = cc[c] = 0.0f;
          if (okc) {ca[c] = bufs.cs[t]; cb[c] = bufs.cs[T + t]; cc[c] = bufs.cs[2 * T + t];}
#pragma unroll
          for (int rr = 0; rr < kRows; ++rr) {
            const int r = seg + (ri0 + rr) * S;
            const bool ok = okc && ri0 + rr < nri && b0 + r < B;
            oo[c][rr] = ok ? t * kPad + r : -1;
            va[c][rr] = vb[c][rr] = vc[c][rr] = 0.0f;
            if (ok) {
              const size_t g = static_cast<size_t>(b0 + r) * T + t;
              va[c][rr] = __ldg(bufs.in_a + g); vb[c][rr] = __ldg(bufs.in_b + g); vc[c][rr] = __ldg(bufs.in_c + g);
            }
          }
        }
#pragma unroll
        for (int c = 0; c < kCols; ++c) {
#pragma unroll
          for (int rr = 0; rr < kRows; ++rr) {
            if (oo[c][rr] >= 0) {
              s_cvx[oo[c][rr]] = __fadd_rn(ca[c], va[c][rr]);
              s_cvy[oo[c][rr]] = __fadd_rn(cb[c], vb[c][rr]);
              s_cwz[oo[c][rr]] = __fadd_rn(cc[c], vc[c][rr]);
            }
          }
        }
      }
    }
  }
  MPPI_TRACE_AT(1);
  if (tid < kHotBytes / 16) {reinterpret_cast<float4 *>(s_hot)[tid] = hot_v;}
  for (int i = tid + nthreads; i < kHotBytes / 16; i += nthreads) {reinterpret_cast<float4 *>(s_hot)[i] = __ldg(hot_src + i);}
  if (tid < 3 * T) {s_cs[tid] = cs_v[0];}
  if (tid + nthreads < 3 * T) {s_cs[tid + nthreads] = cs_v[1];}
  for (int i = tid + 2 * nthreads; i < 3 * T; i += nthreads) {s_cs[i] = bufs.cs[i];}
  __syncthreads();
  MPPI_TRACE_AT(2);
  const bool hol = MPPI_SF(SF_HOL, p.holonomic != 0);
  const bool acker = MPPI_SF(SF_ACKER, p.model == MPPI_MODEL_ACKERMANN);
  const bool con_on = MPPI_SF(SF_CON, p.constraint.on), fwd_on = MPPI_SF(SF_FWD, p.forward.on);
  const bool twirl_on = MPPI_SF(SF_TWIRL, p.twirl.on), db_on = MPPI_SF(SF_DB, p.deadband.on);
  const bool goal_on = MPPI_SF(SF_GOAL, p.goal.on), gang_on = MPPI_SF(SF_GANG, p.goal_angle.on);
  const bool cost_on = MPPI_SF(SF_COST, p.cost.on), ob_on = MPPI_SF(SF_OBST, p.obst.on);
  constexpr bool kFp = (F & SF_FOOTPRINT) != 0, kSpill = (F & SF_SPILL) != 0;
  const float dt = p.dt;
  if (mode == 0) {
    // updateInitialStateVelocities (optimizer.cpp:258-267): v[:,0] = robot speed.  Written and read by warp 0 only
    // (yaw scan, first segment), lane to lane: no barrier
    if (seg == 0) {
      s_v0[lane] = p.speed_vx; s_v0[kTile + lane] = hol ? p.speed_vy : 0.0f; s_v0[2 * kTile + lane] = p.speed_wz;
    }
  } else {
    for (int r = seg; r < kTile; r += S) {
      const int rb = b0 + r;
      if (rb < B) {
        const size_t row = static_cast<size_t>(rb) * T;
        for (int t = lane; t < T; t += 32) {
          const float a = __ldg(bufs.in_a + row + t), bb = __ldg(bufs.in_b + row + t), c = __ldg(bufs.in_c + row + t);
          // injected state velocities: v[t] is stored where predict() would read it, c[t-1]
          if (t == 0) {
            s_v0[r] = a; s_v0[kTile + r] = bb; s_v0[2 * kTile + r] = c;
          } else {
            s_cvx[(t - 1) * kPad + r] = a; s_cvy[(t - 1) * kPad + r] = bb; s_cwz[(t - 1) * kPad + r] = c;
          }
          if (mode == 2) {
            s_x[t * kPad + r] = __ldg(bufs.in_x + row + t);
            s_y[t * kPad + r] = __ldg(bufs.in_y + row + t);
            s_yaw[t * kPad + r] = __ldg(bufs.in_yaw + row + t);
          }
        }
      }
    }
    if (seg == 0 && live) {
      const int o = (T - 1) * kPad + lane;
      s_cvx[o] = 0.0f; s_cvy[o] = 0.0f; s_cwz[o] = 0.0f;
    }
    __syncthreads();
  }

  MPPI_TRACE_AT(3);
  // my segment of the horizon, and the state velocities just before it (read before anyone overwrites a plane)
  const int L = (T + S - 1) / S;
  const int t0 = min(T, seg * L), t1 = min(T, t0 + L);
  const bool use_vy = hol || mode != 0;
  float pvx = 0.0f, pvy = 0.0f, pwz = 0.0f;
  if (live && t0 < t1) {
    if (t0 == 0) {
      pvx = s_v0[lane]; pvy = s_v0[kTile + lane]; pwz = s_v0[2 * kTile + lane];
    } else {
      const int o = (t0 - 1) * kPad + lane;
      pvx = s_cvx[o]; pvy = s_cvy[o]; pwz = s_cwz[o];
    }
    if (!use_vy) {pvy = 0.0f;}
  }

  // ---- P2: yaw = cumsum(wz * dt) + yaw0, sequential in t (optimizer.cpp:319-320)
  if (mode != 2 && seg == 0 && live) {
    // chunks of 8: the eight loads are independent (pipelined), only the eight adds form the carried chain
    const float yaw0 = p.yaw0;
    float acc = -0.0f;                       // (-0) + x == x bit for bit: the first element of the cumsum is the term itself
    float wz = s_v0[2 * kTile + lane];
    for (int tc = 0; tc < T; tc += 8) {
      float w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {w[u] = s_cwz[min(tc + u, T - 1) * kPad + lane];}
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        acc = __fadd_rn(acc, __fmul_rn(wz, dt));
        wz = w[u];
        if (tc + u < T) {s_yaw[(tc + u) * kPad + lane] = __fadd_rn(acc, yaw0);}
      }
    }
  }
  if (kFused) {
    if (zero_copy && up_tid >= 0) {
      uint4 * dst = reinterpret_cast<uint4 *>(const_cast<DevParams *>(P));
      if (up_begin + up_tid < up_end) {dst[up_begin + up_tid] = up_v[0];}
      if (up_begin + up_n + up_tid < up_end) {dst[up_begin + up_n + up_tid] = up_v[1];}
      for (int i = up_begin + 2 * up_n + up_tid; i < up_end; i += up_n) {dst[i] = __ldg(fx->up_host + i);}
      __threadfence();   // this thread's part of the upload slice is visible device-wide ...
    }
  }
  __syncthreads();
  if (kFused) {
    // ... before the tile's flag goes out.  The flag's writer fences too: its fence is cumulative over what the barrier
    // above made visible to it, which is what makes {slice stores, flag} a release in the PTX memory model
    if (zero_copy && tid == 0) {__threadfence(); st_packet(bufs.pk_up + tile, 1u, fx->tag);}
  }

  MPPI_TRACE_AT(4);
  // ---- P3: velocity critics + gamma term, then dx*dt / dy*dt with the one-step yaw lag written in place
  float acc[A_COUNT];
#pragma unroll
  for (int k = 0; k < A_COUNT; ++k) {acc[k] = 0.0f;}
  if (live) {
    const float max_vel = p.max_vel, min_vel = p.min_vel, min_r = p.min_turning_r;
    const float db_vx = fabsf(p.db_vx), db_vy = fabsf(p.db_vy), db_wz = fabsf(p.db_wz);
    float g_vx = 0.0f, g_vy = 0.0f, g_wz = 0.0f, a_con = 0.0f, a_fwd = 0.0f, a_twirl = 0.0f, a_db = 0.0f;
    // steps of the segment in chunks of kTileChunk: the sincos chains of a chunk are independent and overlap (ILP)
    constexpr int kC = kTileChunk;
    for (int tc = t0; tc < t1; tc += kC) {
      float cx[kC], cy[kC], cw[kC], sn[kC], cn[kC];
#pragma unroll
      for (int u = 0; u < kC; ++u) {
        const int o = min(tc + u, t1 - 1) * kPad + lane;
        cx[u] = s_cvx[o]; cy[u] = s_cvy[o]; cw[u] = s_cwz[o];   // controls of step t (state velocities of t+1)
      }
      if (mode != 2) {
        // integrateStateVelocities (optimizer.cpp:322-337): cos/sin of yaw[t-1]
#pragma unroll
        for (int u = 0; u < kC; ++u) {
          const int t = min(tc + u, t1 - 1);
          if (t == 0) {
            sn[u] = p.sin0; cn[u] = p.cos0;
          } else {
            mppi_det_sincosf(s_yaw[(t - 1) * kPad + lane], &sn[u], &cn[u]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kC; ++u) {
        const int t = tc + u;
        if (t < t1) {
          const int o = t * kPad + lane;
          const float vx = pvx, vy = pvy, wz = pwz;                   // state velocities of step t
          if (mode == 0) {
            // gamma term of updateControlSequence (optimizer.cpp:365-380): sum_t cs[t] * (c[b,t] - cs[t])
            const float csx = s_cs[t], csy = s_cs[T + t], csw = s_cs[2 * T + t];
            g_vx = fmaf(csx, __fsub_rn(cx[u], csx), g_vx);
            g_wz = fmaf(csw, __fsub_rn(cw[u], csw), g_wz);
            if (hol) {g_vy = fmaf(csy, __fsub_rn(cy[u], csy), g_vy);}
          }
          if (con_on) {   // constraint_critic.cpp:49-52
            const float sgn = vx > 0.0f ? 1.0f : -1.0f;
            const float vel_total = sgn * sqrt_approx(vx * vx + vy * vy);
            float e = fmaxf(vel_total - max_vel, 0.0f) + fmaxf(min_vel - vel_total, 0.0f);
            if (acker) {e += fmaxf(min_r - fabsf(vx) / fabsf(wz), 0.0f);}
            a_con += e * dt;
          }
          if (fwd_on) {a_fwd += fmaxf(-vx, 0.0f) * dt;}           // prefer_forward_critic.cpp:42-46
          if (twirl_on) {a_twirl += fabsf(wz);}                   // twirling_critic.cpp:40-41
          if (db_on) {                                            // velocity_deadband_critic.cpp:54-97
            float e = fmaxf(db_vx - fabsf(vx), 0.0f);
            if (hol) {e += fmaxf(db_vy - fabsf(vy), 0.0f);}
            e += fmaxf(db_wz - fabsf(wz), 0.0f);
            a_db += e * dt;
          }
          if (mode != 2) {
            float dx = __fmul_rn(vx, cn[u]);
            float dy = __fmul_rn(vx, sn[u]);
            if (hol) {
              dx = __fsub_rn(dx, __fmul_rn(vy, sn[u]));
              dy = __fadd_rn(dy, __fmul_rn(vy, cn[u]));
            }
            s_x[o] = __fmul_rn(dx, dt);    // in place over the control planes: (cx, cy) already live in registers
            s_y[o] = __fmul_rn(dy, dt);
          }
          pvx = cx[u]; pvy = use_vy ? cy[u] : 0.0f; pwz = cw[u];
        }
      }
    }
    acc[A_GVX] = g_vx; acc[A_GVY] = g_vy; acc[A_GWZ] = g_wz;
    acc[A_CON] = a_con; acc[A_FWD] = a_fwd; acc[A_TWIRL] = a_twirl; acc[A_DB] = a_db;
  }

  MPPI_TRACE_AT(5);
  if (mode != 2) {
    __syncthreads();
    // ---- P4: x = pose.x (double) + cumsum(dx*dt) (float), sequential in t (optimizer.cpp:339-342)
    if (live && seg < 2) {
      const bool do_x = seg == 0, do_y = (S > 1) ? (seg == 1) : true;
      // one plane per warp (x: warp 0, y: warp 1), chunks of 8 as above; the fp64 pose add is off the carried chain
      auto scan_plane = [&](float * plane, const double origin) {
          float a = -0.0f;
          for (int tc = 0; tc < T; tc += 8) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {v[u] = plane[min(tc + u, T - 1) * kPad + lane];}
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              a = __fadd_rn(a, v[u]);
              if (tc + u < T) {plane[(tc + u) * kPad + lane] = static_cast<float>(origin + static_cast<double>(a));}
            }
          }
        };
      if (do_x) {scan_plane(s_x, p.pose_x);}
      if (do_y) {scan_plane(s_y, p.pose_y);}
    }
    if (kFused) {
      // zero-copy upload: a warp that has no scan to do collects the flags of all tiles; behind the barrier below the
      // device copies of the record and the costmap are complete
      if (zero_copy && seg == min(2, S - 1)) {
        for (int i = lane; i < ntiles; i += 32) {
          unsigned v;
          if (!poll_packet(bufs.pk_up + i, fx->tag, v)) {raise_comm_error(bufs);}
        }
        __threadfence();   // acquire side: the (coherent) loads of record tail and costmap behind the barrier below see the slices
      }
    }
  }
  __syncthreads();

  MPPI_TRACE_AT(6);
  // fused: the path and its host-made tables (record tail, build_params: x[N] y[N] yaw[N] D[N] | valid[n16] flags[n16]
  // follow[N]) are requested now and committed to shared memory behind the position critics, when they have long arrived
  float pt_f[3] = {0.0f, 0.0f, 0.0f};
  unsigned pt_b = 0u;
  if (kFused) {
    const int N = min(p.N, fx->n_cap), n16 = ((N + 15) / 16) * 16;
    const float * tail = reinterpret_cast<const float *>(P + 1);
    const uint8_t * g_valid = reinterpret_cast<const uint8_t *>(tail + 4 * N);
    const uint16_t * g_follow = reinterpret_cast<const uint16_t *>(g_valid + 2 * n16);
    if (tid < N) {
      pt_f[0] = ld_ro<kNc>(tail + 3 * N + tid); pt_f[1] = ld_ro<kNc>(tail + tid); pt_f[2] = ld_ro<kNc>(tail + N + tid);
      pt_b = ld_ro<kNc>(g_valid + tid) | (static_cast<unsigned>(ld_ro<kNc>(g_valid + n16 + tid)) << 8) |
        (static_cast<unsigned>(ld_ro<kNc>(g_follow + tid)) << 16);
    }
  }
  // ---- P5: position critics + spills, parallel over (trajectory, segment of the horizon)
  if (live) {
    const bool want_cells = kSpill && p.want_cells != 0, spill = kSpill && p.spill_traj != 0;
    const bool need_cell = cost_on || ob_on || want_cells;
    const bool track_unknown = p.track_unknown != 0;
    const bool cost_fp = kFp && p.cost_fp != 0, ob_fp = kFp && p.obst_fp != 0;
    const bool cost_near_goal = p.cost_near_goal != 0, ob_near_goal = p.obst_near_goal != 0, ob_rep_on = p.obst_repulsion_enabled != 0;
    const float cost_pic = p.cost_possibly_inscribed, ob_pic = p.obst_possibly_inscribed, cost_critical = p.cost_critical;
    const double gx = p.goal_x, gy = p.goal_y, ox = p.ox, oy = p.oy, res = p.res;
    const unsigned size_x = p.size_x, size_y = p.size_y;
    const CellGrid cg = {p.cell_oxf, p.cell_oyf, p.cell_invf, 0.5f - p.cell_eps_x, 0.5f - p.cell_eps_y, size_x, size_y};
    const float goal_yaw = p.goal_yaw;
    const int step = p.sample_step;
    int next_sample = T, sample_k = 0;
    if (step > 0) {sample_k = (t0 + step - 1) / step; next_sample = sample_k * step;}
    const bool sample_yaw = p.sample_yaw != 0;
    bool cost_hit = false, ob_hit = false;
    float a_goal = 0.0f, a_gang = 0.0f, cost_rep = 0.0f, ob_traj = 0.0f, ob_rep = 0.0f;
    size_t g = static_cast<size_t>(t0) * B + b;
    // steps of the segment in chunks of kTileChunk: the cell indices are computed and their costmap bytes requested
    // together (one memory round trip per chunk instead of one per step); the collision logic stays in step order
    constexpr int kC = kTileChunk;
    for (int tc = t0; tc < t1; tc += kC) {
      float pxs[kC], pys[kC];
      int cells[kC], pcs[kC];
#pragma unroll
      for (int u = 0; u < kC; ++u) {
        const int oo = min(tc + u, t1 - 1) * kPad + lane;
        pxs[u] = s_x[oo]; pys[u] = s_y[oo];
      }
      if (need_cell) {
#pragma unroll
        for (int u = 0; u < kC; ++u) {cells[u] = world_to_cell_fast(pxs[u], pys[u], cg, &p.res);}
#pragma unroll
        for (int u = 0; u < kC; ++u) {pcs[u] = cells[u] < 0 ? NO_INFORMATION : ld_ro<kNc>(cm + cells[u]);}
      }
#pragma unroll
      for (int u = 0; u < kC; ++u) {
        const int t = tc + u;
        if (t >= t1) {break;}
        const int o = t * kPad + lane;
        const float px = pxs[u], py = pys[u];
        if (goal_on) {                                               // goal_critic.cpp:50-52
          const float dx = static_cast<float>(static_cast<double>(px) - gx);
          const float dy = static_cast<float>(static_cast<double>(py) - gy);
          a_goal += sqrt_approx(dx * dx + dy * dy);
        }
        if (gang_on) {                                               // goal_angle_critic.cpp:47-49
          a_gang += static_cast<float>(fabs(normalize_angle_d(static_cast<double>(__fsub_rn(goal_yaw, s_yaw[o])))));
        }
        if (need_cell) {
          const int cell = cells[u];
          if (want_cells) {bufs.spill_cells[g] = cell;}
          if ((cost_on && !cost_hit) || (ob_on && !ob_hit)) {
            const int pose_cost = pcs[u];
            int fp_cost = -1;
            if (cost_on && !cost_hit && pose_cost >= 1) {            // cost_critic.cpp:139-162
              int c = pose_cost;
              if (cost_fp && (static_cast<float>(c) >= cost_pic || cost_pic < 1.0f)) {
                fp_cost = footprint_cost_at_pose<kNc>(P, p.fp_n, ox, oy, res, size_x, size_y, cm, px, py, s_yaw[o]);
                c = fp_cost;
              }
              if (in_collision(c, cost_fp, track_unknown)) {
                cost_hit = true;
              } else if (pose_cost >= INSCRIBED_INFLATED_OBSTACLE) {
                cost_rep += cost_critical;
              } else if (!cost_near_goal) {
                cost_rep += static_cast<float>(pose_cost);
              }
            }
            if (ob_on && !ob_hit) {                                  // obstacles_critic.cpp:145-170, :203-224
              int c = pose_cost;
              int using_fp = 0;
              if (cell >= 0 && ob_fp && (static_cast<float>(c) >= ob_pic || ob_pic < 1.0f)) {
                if (fp_cost < 0) {fp_cost = footprint_cost_at_pose<kNc>(P, p.fp_n, ox, oy, res, size_x, size_y, cm, px, py, s_yaw[o]);}
                c = fp_cost;
                using_fp = 1;
              }
              if (c >= 1) {
                if (in_collision(c, ob_fp, track_unknown)) {
                  ob_hit = true;
                } else if (ob_rep_on) {
                  ob_traj += ld_ro<kNc>(&P->obst_lut_crit[using_fp][c]);
                  if (!ob_near_goal) {ob_rep += ld_ro<kNc>(&P->obst_lut_rep[using_fp][c]);}
                }
              }
            }
          }
        }
        // spills for the path critics of K3 (the fused tail reads the poses straight from the tile)
        if (!kFused && t == next_sample) {
          const size_t k = static_cast<size_t>(sample_k) * B + b;
          bufs.samples_x[k] = px;
          bufs.samples_y[k] = py;
          if (sample_yaw) {bufs.samples_yaw[k] = s_yaw[o];}
          next_sample += step; sample_k++;
        }
        if (spill) {
          bufs.spill_x[g] = px; bufs.spill_y[g] = py; bufs.spill_yaw[g] = s_yaw[o];
        }
        if (kSpill && p.vis_b_step > 0 && t % p.vis_t_step == 0 && b % p.vis_b_step == 0) {
          // TrajectoryVisualizer::add (trajectory_visualizer.cpp:86-108) reads only this lattice of the candidates
          const int nt = (T + p.vis_t_step - 1) / p.vis_t_step;
          const size_t k = static_cast<size_t>(t / p.vis_t_step) * p.vis_nb + b / p.vis_b_step;
          bufs.vis_xy[k] = px; bufs.vis_xy[static_cast<size_t>(nt) * p.vis_nb + k] = py;
        }
        g += B;
      }
    }
    if (!kFused && t1 == T && t0 < t1) {
      bufs.end_xy[b] = s_x[(T - 1) * kPad + lane];
      bufs.end_xy[B + b] = s_y[(T - 1) * kPad + lane];
    }
    acc[A_GOAL] = a_goal; acc[A_GANG] = a_gang; acc[A_COST_REP] = cost_rep; acc[A_OB_TRAJ] = ob_traj; acc[A_OB_REP] = ob_rep;
    acc[A_COST_HIT] = cost_hit ? 1.0f : 0.0f;
    acc[A_OB_HIT] = ob_hit ? 1.0f : 0.0f;
  }
#pragma unroll
  for (int k = 0; k < A_COUNT; ++k) {s_acc[(seg * A_COUNT + k) * kTile + lane] = acc[k];}
  if (kFused) {
    const int N = min(p.N, fx->n_cap), n16 = ((N + 15) / 16) * 16;
    if (tid < N) {
      fs.D[tid] = pt_f[0]; fs.px[tid] = pt_f[1]; fs.py[tid] = pt_f[2];
      fs.valid[tid] = static_cast<uint8_t>(pt_b & 0xffu); fs.flags[tid] = static_cast<uint8_t>((pt_b >> 8) & 0xffu);
      fs.follow[tid] = static_cast<uint16_t>(pt_b >> 16);
    }
    // paths longer than the block: plain loop (rare)
    const float * tail = reinterpret_cast<const float *>(P + 1);
    const uint8_t * g_valid = reinterpret_cast<const uint8_t *>(tail + 4 * N);
    const uint16_t * g_follow = reinterpret_cast<const uint16_t *>(g_valid + 2 * n16);
    for (int j = tid + nthreads; j < N; j += nthreads) {
      fs.D[j] = ld_ro<kNc>(tail + 3 * N + j); fs.px[j] = ld_ro<kNc>(tail + j); fs.py[j] = ld_ro<kNc>(tail + N + j);
      fs.valid[j] = ld_ro<kNc>(g_valid + j); fs.flags[j] = ld_ro<kNc>(g_valid + n16 + j); fs.follow[j] = ld_ro<kNc>(g_follow + j);
    }
  }

  MPPI_TRACE_AT(7);
  // ---- furthest reached path point candidate: argmin over the path of the end pose (utils.hpp:292-319),
  //      path range split over the warps, combined in order so the first minimum wins
  const int N = p.N;
  const bool need_furthest = p.need_furthest != 0;
  if (need_furthest) {
    const float * path_x = reinterpret_cast<const float *>(P + 1) + p.off_path_x;
    const float * path_y = reinterpret_cast<const float *>(P + 1) + p.off_path_y;
    const float ex = s_x[(T - 1) * kPad + lane], ey = s_y[(T - 1) * kPad + lane];
    const int per = (N + S - 1) / S;
    const int j0 = seg * per, j1 = min(N, j0 + per);
    float best = 3.402823466e+38f;
    int best_j = j0 < N ? j0 : 0;
    for (int j = j0; j < j1; ++j) {
      const float dx = __fsub_rn(ld_ro<kNc>(path_x + j), ex);
      const float dy = __fsub_rn(ld_ro<kNc>(path_y + j), ey);
      const float d = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
      if (d < best) {best = d; best_j = j;}
    }
    s_amin_d[seg * kTile + lane] = best;
    s_amin_j[seg * kTile + lane] = best_j;
  }
  __syncthreads();

  MPPI_TRACE_AT(8);
  // ---- P6: combine the segments in order and finish the per-critic terms: accumulator k (and the critic row it feeds)
  //      by warp k mod S, lane = trajectory; the collision flags gate the sums they belong to.  The furthest-point
  //      candidate is combined by the last warp.  Nothing here is serial over the critics.
  {
    const float Tf = static_cast<float>(T);
    float * rows = bufs.crit_rows;
    // a row goes to global memory for K3 (and the per-critic getter); the fused tail takes it from shared memory
    const bool rows_to_global = !kFused || p.want_critic_rows != 0;
    auto put = [&](int q, float v) {
        if (live) {
          if (kFused) {fs.rows[q * kTile + lane] = v;}
          if (rows_to_global) {rows[static_cast<size_t>(q) * B + b] = v;}
        }
      };
    const float * a0 = s_acc + lane;   // [s][k][32]
    unsigned my_flags = 0u;            // fused: bit 16 = a trajectory of this tile survived the Cost critic, bit 17 = Obstacles
    for (int k = seg; k < A_COUNT; k += S) {
      if (k == A_COST_HIT || k == A_OB_REP || k == A_OB_HIT) {continue;}   // combined with the sums they gate
      if (k <= A_GWZ) {
        float t = a0[k * kTile];
        for (int s = 1; s < S; ++s) {t = __fadd_rn(t, a0[(s * A_COUNT + k) * kTile]);}
        switch (k) {
          case A_CON: if (con_on) {put(p.constraint.idx, add_pow_c(0.0f, t * p.constraint.weight, p.constraint.power));} break;
          case A_FWD: if (fwd_on) {put(p.forward.idx, add_pow_c(0.0f, t * p.forward.weight, p.forward.power));} break;
          case A_TWIRL: if (twirl_on) {put(p.twirl.idx, add_pow_c(0.0f, (t / Tf) * p.twirl.weight, p.twirl.power));} break;
          case A_DB: if (db_on) {put(p.deadband.idx, add_pow_c(0.0f, t * p.deadband.weight, p.deadband.power));} break;
          case A_GOAL: if (goal_on) {put(p.goal.idx, add_pow_c(0.0f, (t / Tf) * p.goal.weight, p.goal.power));} break;
          case A_GANG: if (gang_on) {put(p.goal_angle.idx, add_pow_c(0.0f, (t / Tf) * p.goal_angle.weight, p.goal_angle.power));} break;
          case A_GVX: if (mode == 0) {put(p.n_critics, t);} break;
          case A_GVY: if (mode == 0) {put(p.n_critics + 1, t);} break;
          default: if (mode == 0) {put(p.n_critics + 2, t);} break;   // A_GWZ
        }
      } else if (k == A_COST_REP) {
        if (cost_on) {   // cost_critic.cpp:159-166
          float t = 0.0f;
          bool hit = false;
          for (int s = 0; s < S && !hit; ++s) {
            t += a0[(s * A_COUNT + A_COST_REP) * kTile];
            hit = a0[(s * A_COUNT + A_COST_HIT) * kTile] != 0.0f;
          }
          const float rep = hit ? p.cost_collision : t;
          put(p.cost.idx, add_pow_c(0.0f, p.cost.weight * rep / Tf, p.cost.power));
          // fail_flag input: did any trajectory of this tile survive?
          const unsigned ok = __ballot_sync(0xffffffffu, live && !hit);
          if (kFused) {
            if (ok) {my_flags |= 0x10000u;}
          } else if (lane == 0 && ok) {
            atomicOr(&bufs.st->any_ok[p.cost.idx], 1u);
          }
        }
      } else {   // A_OB_TRAJ (+ A_OB_REP, A_OB_HIT)
        if (ob_on) {   // obstacles_critic.cpp:169-176
          float t = 0.0f, rp = 0.0f;
          bool hit = false;
          for (int s = 0; s < S && !hit; ++s) {
            t += a0[(s * A_COUNT + A_OB_TRAJ) * kTile];
            rp += a0[(s * A_COUNT + A_OB_REP) * kTile];
            hit = a0[(s * A_COUNT + A_OB_HIT) * kTile] != 0.0f;
          }
          const float raw = hit ? p.obst_collision : t;
          put(p.obst.idx, add_pow_c(0.0f, (p.obst_critical_w * raw) + (p.obst_repulsion_w * rp / Tf), p.obst.power));
          const unsigned ok = __ballot_sync(0xffffffffu, live && !hit);
          if (kFused) {
            if (ok) {my_flags |= 0x20000u;}
          } else if (lane == 0 && ok) {
            atomicOr(&bufs.st->any_ok[p.obst.idx], 1u);
          }
        }
      }
    }
    // this tile's furthest-point candidate: the segments' minima combined in order so the first minimum wins
    if (seg == S - 1 && need_furthest) {
      float best = s_amin_d[lane];
      int best_j = s_amin_j[lane];
      for (int s = 1; s < S; ++s) {
        const float d = s_amin_d[s * kTile + lane];
        if (d < best) {best = d; best_j = s_amin_j[s * kTile + lane];}
      }
      const unsigned cand = warp_max_u(live ? static_cast<unsigned>(best_j) : 0u);
      if (kFused) {
        my_flags |= cand;   // path indices are < MPPI_MAX_PATH_POINTS <= 2^16
      } else if (lane == 0) {
        atomicMax(&bufs.st->furthest_candidate, cand);
      }
    }
    if (kFused) {
      // exchange 1 inside the GPU: one self-validating packet per tile {candidate | survivor flags << 16, tag}, put
      // together from the warps that own the pieces
      unsigned * s_x1 = reinterpret_cast<unsigned *>(fs.stat) + 7;   // zeroed at kernel start
      if (lane == 0 && my_flags) {atomicOr(s_x1, my_flags);}
      __syncthreads();         // also publishes fs.rows to the tail
      if (tid == 0) {st_packet(bufs.pk_x1 + tile, *s_x1, fx->tag);}
    }
  }
  MPPI_TRACE_AT(9);
}

// kDevMap: the cycle's costmap is the caller's device memory, whose pointer the record carries (DevParams::cm_dev), so that
// a replayed graph reads the pointer of every cycle; cm is not used then.  Separate instances, so that the host-map
// instances stay the code they are.
template<unsigned F, bool kExact, int kMode, bool kDevMap = false>
__global__ void __launch_bounds__(256, MPPI_K2_MIN_BLOCKS) rollout_score_kernel(
  const DevParams * __restrict__ P, const uint8_t * __restrict__ cm, DevBuffers bufs, const int B, const int T)
{
  rollout_tile_body<F, kExact, kMode, false>(P, kDevMap ? P->cm_dev : cm, bufs, B, T, nullptr);
}

// ---------------------------------------------------------------------------------------------------
// K2, stream variant (large batches): one thread owns one trajectory for the whole horizon and everything
// lives in registers.  The noise planes are stored TIME-MAJOR [T][B] for this variant, so lane == trajectory
// reads are coalesced straight from HBM/L2 with no shared-memory staging, no transposes and no barriers.
// The horizon is walked in chunks of kStreamChunk steps; inside a chunk the work is phased so that the
// expensive, mutually independent parts (sincos of the lagged yaw, fp64 cell index, costmap byte gather)
// of the chunk's steps are issued back to back (instruction-level parallelism within one thread), while the
// three cumulative sums stay strictly sequential in t.  Arithmetic (order of the sums, non-contractable fp32
// ops, fp64 index math) is identical to the tile variant and to the oracle.
// The template mask removes whole critic families at compile time (smaller code, fewer registers); every
// family that is compiled in is still gated by its per-cycle runtime flag.
// ---------------------------------------------------------------------------------------------------

constexpr int kStreamThreads = 128;    // upper bound of the block size (the host may launch fewer threads per block)
#ifndef MPPI_STREAM_CHUNK
#define MPPI_STREAM_CHUNK 4
#endif
constexpr int kStreamChunk = MPPI_STREAM_CHUNK;   // steps per phase group == noise rows in flight per thread
constexpr int kNoisePadRows = 8;       // rows allocated behind every noise plane so that the prefetch needs no clamp
static_assert(kStreamChunk <= kNoisePadRows, "prefetch reads up to kStreamChunk rows past the horizon");
#ifndef MPPI_STREAM_MIN_BLOCKS
#define MPPI_STREAM_MIN_BLOCKS 4
#endif

// kExact: the mask IS the set of active features (no runtime flag tests inside the loop); otherwise the mask is an
// upper bound and every feature is still gated by its per-cycle runtime flag (generic instance).
// nblocks: a block at or beyond it returns at once (a robot-group member in a launch sized for a larger member); the
// check sits behind the PDL trigger, where it leaves the kernel's register allocation as it is without it
template<unsigned F, bool kExact>
__device__ __forceinline__ void rollout_score_stream_body(
  const DevParams * __restrict__ P, const uint8_t * __restrict__ cm, const DevBuffers & bufs, int nblocks = 0x7fffffff)
{
  extern __shared__ float smem[];
  const int tid = threadIdx.x;
  const int nthr = blockDim.x;
  pdl_launch_dependents();   // the path-cost kernel behind this one may stage its tables while this grid drains
  if (static_cast<int>(blockIdx.x) >= nblocks) {return;}
  float * s_hot = smem;
  load_hot_params(s_hot, P, tid, nthr);
  __syncthreads();
  const DevParams & p = *reinterpret_cast<const DevParams *>(s_hot);
  const int T = p.T, B = p.B;
  const int Tp = ((T + kStreamChunk - 1) / kStreamChunk) * kStreamChunk;   // horizon padded to whole chunks
  float * s_cs = s_hot + kHotFloats;   // [3][Tp], zero padded
  float * s_fp = s_cs + 3 * Tp;        // [threads][3]: per warp 32 slots {x, y, yaw} for the compacted footprint checks
  for (int t = tid; t < Tp; t += nthr) {
    const bool in = t < T;
    s_cs[t] = in ? bufs.cs[t] : 0.0f;
    s_cs[Tp + t] = in ? bufs.cs[T + t] : 0.0f;
    s_cs[2 * Tp + t] = in ? bufs.cs[2 * T + t] : 0.0f;
  }
  __syncthreads();

  const int b = blockIdx.x * nthr + tid;
  const bool live = b < B;
  const unsigned bb = live ? b : B - 1;  // dead lanes shadow the last trajectory (no divergence, no stores)
  const float dt = p.dt;
  const float * __restrict__ nvx = bufs.in_a;
  const float * __restrict__ nvy = bufs.in_b;
  const float * __restrict__ nwz = bufs.in_c;

  const bool hol = MPPI_SF(SF_HOL, p.holonomic != 0);
  const bool acker = MPPI_SF(SF_ACKER, p.model == MPPI_MODEL_ACKERMANN);
  const bool con_on = MPPI_SF(SF_CON, p.constraint.on), fwd_on = MPPI_SF(SF_FWD, p.forward.on);
  const bool twirl_on = MPPI_SF(SF_TWIRL, p.twirl.on), db_on = MPPI_SF(SF_DB, p.deadband.on);
  const bool goal_on = MPPI_SF(SF_GOAL, p.goal.on), gang_on = MPPI_SF(SF_GANG, p.goal_angle.on);
  const bool cost_on = MPPI_SF(SF_COST, p.cost.on), ob_on = MPPI_SF(SF_OBST, p.obst.on);
  constexpr bool kFp = (F & SF_FOOTPRINT) != 0, kSpill = (F & SF_SPILL) != 0;
  const bool cost_fp = kFp && p.cost_fp != 0, ob_fp = kFp && p.obst_fp != 0;
  const bool want_cells = kSpill && p.want_cells != 0, spill = kSpill && p.spill_traj != 0;
  const bool need_cell = cost_on || ob_on || want_cells;
  const bool track_unknown = p.track_unknown != 0;
  const bool cost_near_goal = p.cost_near_goal != 0, ob_near_goal = p.obst_near_goal != 0, ob_rep_on = p.obst_repulsion_enabled != 0;
  const float cost_pic = p.cost_possibly_inscribed, ob_pic = p.obst_possibly_inscribed, cost_critical = p.cost_critical;
  const float max_vel = p.max_vel, min_vel = p.min_vel, min_r = p.min_turning_r;
  const float db_vx = fabsf(p.db_vx), db_vy = fabsf(p.db_vy), db_wz = fabsf(p.db_wz);
  const double x0 = p.pose_x, y0 = p.pose_y;
  const CellGrid cg = {p.cell_oxf, p.cell_oyf, p.cell_invf, 0.5f - p.cell_eps_x, 0.5f - p.cell_eps_y, p.size_x, p.size_y};
  const float yaw0 = p.yaw0, goal_yaw = p.goal_yaw;
  const int step = p.sample_step;
  const bool sample_yaw = p.sample_yaw != 0;
  const bool step_is_chunk = step == kStreamChunk;

  float g_vx = 0.f, g_vy = 0.f, g_wz = 0.f, a_con = 0.f, a_fwd = 0.f, a_twirl = 0.f, a_db = 0.f;
  float a_goal = 0.f, a_gang = 0.f, cost_rep = 0.f, ob_traj = 0.f, ob_rep = 0.f;
  bool cost_hit = false, ob_hit = false;
  float vx = p.speed_vx, vy = hol ? p.speed_vy : 0.0f, wz = p.speed_wz;   // state velocities of step 0 = robot speed
  // the running sums start at -0.0f: (-0) + x == x bit for bit, i.e. the first element of the cumsum is the term itself
  float acc_yaw = -0.0f, acc_x = -0.0f, acc_y = -0.0f;
  float yaw_prev = yaw0;                 // cos/sin of step 0 use yaw0 (p.cos0 / p.sin0 are mppi_det_sincosf(yaw0) as well)
  float ex = 0.f, ey = 0.f;              // end pose
  int next_sample = step > 0 ? 0 : T;
  unsigned sample_o = 0u;               // element offset of the next PathAlign sample row

  // software pipeline of the noise rows: the chunk being processed was loaded one chunk ago.  32-bit element
  // offsets (the host guarantees (T + pad) * B < 2^32): one IMAD.WIDE per load instead of 64-bit arithmetic.
  float qx[kStreamChunk], qy[kStreamChunk], qw[kStreamChunk];
  unsigned off = bb;                     // element offset of (row, trajectory) in the time-major planes
#pragma unroll
  for (int u = 0; u < kStreamChunk; ++u) {
    qx[u] = __ldg(nvx + off); qw[u] = __ldg(nwz + off);
    qy[u] = hol ? __ldg(nvy + off) : 0.0f;
    off += B;
  }
  unsigned g = b;   // index of (t, b) in the time-major spills

  auto chunk = [&](auto tail_tag, auto step_tag, const int t0) {
      constexpr bool kTail = decltype(tail_tag)::value;   // the last, partial chunk: steps t >= T are masked
      constexpr bool kStepChunk = decltype(step_tag)::value;   // PathAlign samples every kStreamChunk-th pose (the usual step)
      const float * cs_t = s_cs + t0;
      // ---- phase A: noised controls of the chunk (noise_generator.cpp:71-73), then refill the pipeline
      float cx[kStreamChunk], cy[kStreamChunk], cw[kStreamChunk];
#pragma unroll
      for (int u = 0; u < kStreamChunk; ++u) {
        const float csx = cs_t[u], csw = cs_t[2 * Tp + u];
        cx[u] = __fadd_rn(csx, qx[u]);
        cw[u] = __fadd_rn(csw, qw[u]);
        // gamma term (optimizer.cpp:365-380) while the control sequence is at hand; the padded steps of the last chunk
        // carry a zero control sequence and zero noise rows: their terms are exact zeros
        g_vx = fmaf(csx, __fsub_rn(cx[u], csx), g_vx);
        g_wz = fmaf(csw, __fsub_rn(cw[u], csw), g_wz);
        if (hol) {
          const float csy = cs_t[Tp + u];
          cy[u] = __fadd_rn(csy, qy[u]);
          g_vy = fmaf(csy, __fsub_rn(cy[u], csy), g_vy);
        } else {
          cy[u] = 0.0f;
        }
      }
      if (!kTail) {
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {
          qx[u] = __ldg(nvx + off); qw[u] = __ldg(nwz + off);
          qy[u] = hol ? __ldg(nvy + off) : 0.0f;
          off += B;
        }
      }
      // ---- phase B: yaw = cumsum(wz * dt) + yaw0 (optimizer.cpp:319-320), sequential; one add per step
      float yw[kStreamChunk], sn[kStreamChunk], cn[kStreamChunk];
#pragma unroll
      for (int u = 0; u < kStreamChunk; ++u) {
        const float swz = u == 0 ? wz : cw[u - 1];
        acc_yaw = __fadd_rn(acc_yaw, __fmul_rn(swz, dt));
        yw[u] = __fadd_rn(acc_yaw, yaw0);
      }
      // ---- phase C: cos/sin of the lagged yaw (optimizer.cpp:322-329): independent across the chunk
      //      one range test per chunk: yaw angles are small, the large-argument reduction is a branch never taken
      bool small = true;
#pragma unroll
      for (int u = 0; u < kStreamChunk; ++u) {small = small && fabsf(u == 0 ? yaw_prev : yw[u - 1]) <= 1.0e5f;}
      if (small) {
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {mppi_det_sincosf_small(u == 0 ? yaw_prev : yw[u - 1], &sn[u], &cn[u]);}
      } else {
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {mppi_det_sincosf(u == 0 ? yaw_prev : yw[u - 1], &sn[u], &cn[u]);}
      }
      // ---- phase D: x = pose.x + cumsum(dx * dt) (optimizer.cpp:331-342), sequential; fp64 add of the pose
      float px[kStreamChunk], py[kStreamChunk];
#pragma unroll
      for (int u = 0; u < kStreamChunk; ++u) {
        const float svx = u == 0 ? vx : cx[u - 1];
        float dx = __fmul_rn(svx, cn[u]), dy = __fmul_rn(svx, sn[u]);
        if (hol) {
          const float svy = u == 0 ? vy : cy[u - 1];
          dx = __fsub_rn(dx, __fmul_rn(svy, sn[u]));
          dy = __fadd_rn(dy, __fmul_rn(svy, cn[u]));
        }
        acc_x = __fadd_rn(acc_x, __fmul_rn(dx, dt));
        acc_y = __fadd_rn(acc_y, __fmul_rn(dy, dt));
        px[u] = static_cast<float>(x0 + static_cast<double>(acc_x));
        py[u] = static_cast<float>(y0 + static_cast<double>(acc_y));
      }
      // ---- phase E: costmap cell of every pose of the chunk and its byte, loads issued together
      int cell[kStreamChunk], pcost[kStreamChunk];
      bool costed = false;   // some pose of the chunk needs the obstacle-type critics' attention
      if (need_cell) {
        bool all_plain = true;
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {
          bool plain;
          cell[u] = world_to_cell_plain(px[u], py[u], cg, plain);
          all_plain = all_plain && plain;
        }
        int any = 0;
        if (all_plain) {   // every pose of the chunk certainly in its fp32 cell and on the map: the usual case
#pragma unroll
          for (int u = 0; u < kStreamChunk; ++u) {pcost[u] = __ldg(cm + static_cast<unsigned>(cell[u])); any |= pcost[u];}
        } else {           // one branch per chunk: poses off the map, and the reference's own fp64 arithmetic where it decides
#pragma unroll
          for (int u = 0; u < kStreamChunk; ++u) {
            cell[u] = world_to_cell_fast(px[u], py[u], cg, &p.res);
            pcost[u] = cell[u] < 0 ? NO_INFORMATION : __ldg(cm + cell[u]); any |= pcost[u];
          }
        }
        // free space under every pose of the chunk (the common case): nothing for Cost / Obstacles to do - unless the
        // Obstacles critic checks the footprint at every pose (no inflation layer: possibly_inscribed_cost < 1)
        costed = any != 0 || want_cells || (ob_on && ob_fp && ob_pic < 1.0f);
      }
      // ---- phase F1: the critics that do not look at the costmap; straight-line code, independent across the chunk
#pragma unroll
      for (int u = 0; u < kStreamChunk; ++u) {
        const int t = t0 + u;
        if (!kTail || t < T) {
          const float svx = u == 0 ? vx : cx[u - 1];
          const float svy = u == 0 ? vy : cy[u - 1];
          const float swz = u == 0 ? wz : cw[u - 1];
          if (con_on) {   // constraint_critic.cpp:49-52
            const float sgn = svx > 0.0f ? 1.0f : -1.0f;
            const float vel_total = sgn * sqrt_approx(svx * svx + svy * svy);
            float e = fmaxf(vel_total - max_vel, 0.0f) + fmaxf(min_vel - vel_total, 0.0f);
            if (acker) {e += fmaxf(min_r - fabsf(svx) / fabsf(swz), 0.0f);}
            a_con += e * dt;
          }
          if (fwd_on) {a_fwd += fmaxf(-svx, 0.0f) * dt;}       // prefer_forward_critic.cpp:42-46
          if (twirl_on) {a_twirl += fabsf(swz);}               // twirling_critic.cpp:40-41
          if (db_on) {                                         // velocity_deadband_critic.cpp:54-97
            float e = fmaxf(db_vx - fabsf(svx), 0.0f);
            if (hol) {e += fmaxf(db_vy - fabsf(svy), 0.0f);}
            e += fmaxf(db_wz - fabsf(swz), 0.0f);
            a_db += e * dt;
          }
          if (goal_on) {                                       // goal_critic.cpp:50-52
            const float ddx = static_cast<float>(static_cast<double>(px[u]) - p.goal_x);
            const float ddy = static_cast<float>(static_cast<double>(py[u]) - p.goal_y);
            a_goal += sqrt_approx(ddx * ddx + ddy * ddy);
          }
          if (gang_on) {a_gang += static_cast<float>(fabs(normalize_angle_d(static_cast<double>(__fsub_rn(goal_yaw, yw[u])))));}
        }
      }
      // ---- phase F2: Cost / Obstacles, in step order (the collision short-circuits are order dependent); one branch
      //      per chunk: skipped while every pose of the chunk sits in free space
      // Footprint mode: the poses of the chunk whose point cost sends a critic to the footprint check (cost_critic.cpp:204-209,
      // obstacles_critic.cpp:214-220) are collected over the WARP first - 4 poses x 32 lanes, typically a seventh of them in a
      // boxed-in scene - and checked one per lane in as few passes as possible, instead of one divergent call per pose with a
      // handful of lanes active (7 threads per warp instruction in profiles/r02c, 85 % of the kernel's time).  The check is a
      // pure function of the pose, so checking a pose the step-order walk below would have skipped (behind a collision
      // earlier in the SAME chunk) changes nothing; the set collected is a superset of what the walk asks for.
      // Inlined on purpose: out of line (a __noinline__ helper taking the chunk's poses) the call makes the hot loop spill -
      // 236 against 140 us at 262144 x 100, 45 against 32 us at 16384 x 56 (profiles/r02c_compaction_ab.txt).  The price of
      // the inlined form is code that a scene without footprint checks still has to fetch: + 3 us on the COLD 29 us rollout
      // of config 3's literal geometry (nothing warm), + 1 us of 140 us at 262144 x 100.
      int fpc[kStreamChunk];
#pragma unroll
      for (int u = 0; u < kStreamChunk; ++u) {fpc[u] = -1;}
      const bool costed_any = kFp ? __any_sync(0xffffffffu, costed) != 0 : costed;
      if (kFp && costed_any) {
        bool need[kStreamChunk];
        bool need_some = false;
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {
          const float pc = static_cast<float>(pcost[u]);
          const bool nc = cost_on && cost_fp && !cost_hit && pcost[u] >= 1 && (pc >= cost_pic || cost_pic < 1.0f);
          const bool no = ob_on && ob_fp && !ob_hit && cell[u] >= 0 && (pc >= ob_pic || ob_pic < 1.0f);
          need[u] = costed && (!kTail || t0 + u < T) && (nc || no);
          need_some = need_some || need[u];
        }
        if (__any_sync(0xffffffffu, need_some)) {   // warp-uniform; one vote where no pose of the warp needs a check
          const unsigned lane = static_cast<unsigned>(tid) & 31u, lt = (1u << lane) - 1u;
          float * slot = s_fp + (tid & ~31) * 3;
          int j[kStreamChunk];
          int total = 0;
#pragma unroll
          for (int u = 0; u < kStreamChunk; ++u) {
            const unsigned m = __ballot_sync(0xffffffffu, need[u]);
            j[u] = need[u] ? total + __popc(m & lt) : -1;
            total += __popc(m);
          }
          for (int r0 = 0; r0 < total; r0 += 32) {
#pragma unroll
            for (int u = 0; u < kStreamChunk; ++u) {
              const int k = j[u] - r0;
              if (k >= 0 && k < 32) {slot[3 * k] = px[u]; slot[3 * k + 1] = py[u]; slot[3 * k + 2] = yw[u];}
            }
            __syncwarp();
            int res = 0;
            if (r0 + static_cast<int>(lane) < total) {
              res = footprint_cost_at_pose<true>(P, p.fp_n, p.ox, p.oy, p.res, cg.size_x, cg.size_y, cm,
                  slot[3 * lane], slot[3 * lane + 1], slot[3 * lane + 2]);
            }
            __syncwarp();
            slot[3 * lane] = __int_as_float(res);
            __syncwarp();
#pragma unroll
            for (int u = 0; u < kStreamChunk; ++u) {
              const int k = j[u] - r0;
              if (k >= 0 && k < 32) {fpc[u] = __float_as_int(slot[3 * k]);}
            }
            __syncwarp();
          }
        }
      }
      if (costed) {
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {
          const int t = t0 + u;
          if (!kTail || t < T) {
            if (want_cells && live) {bufs.spill_cells[g + static_cast<unsigned>(u) * static_cast<unsigned>(B)] = cell[u];}
            const int pose_cost = pcost[u];
            int fp_cost = -1;
            if (cost_on && !cost_hit && pose_cost >= 1) {   // cost_critic.cpp:139-162
              int c = pose_cost;
              if (kFp && cost_fp && (static_cast<float>(c) >= cost_pic || cost_pic < 1.0f)) {
                fp_cost = fpc[u];
                c = fp_cost;
              }
              if (in_collision(c, cost_fp, track_unknown)) {
                cost_hit = true;
              } else if (pose_cost >= INSCRIBED_INFLATED_OBSTACLE) {
                cost_rep += cost_critical;
              } else if (!cost_near_goal) {
                cost_rep += static_cast<float>(pose_cost);
              }
            }
            if (ob_on && !ob_hit) {                         // obstacles_critic.cpp:145-170, :203-224
              int c = pose_cost;
              int using_fp = 0;
              if (kFp && cell[u] >= 0 && ob_fp && (static_cast<float>(c) >= ob_pic || ob_pic < 1.0f)) {
                fp_cost = fpc[u];
                c = fp_cost;
                using_fp = 1;
              }
              if (c >= 1) {
                if (in_collision(c, ob_fp, track_unknown)) {
                  ob_hit = true;
                } else if (ob_rep_on) {
                  ob_traj += __ldg(&P->obst_lut_crit[using_fp][c]);
                  if (!ob_near_goal) {ob_rep += __ldg(&P->obst_lut_rep[using_fp][c]);}
                }
              }
            }
          }
        }
      }
      // ---- phase F3: what leaves the kernel per pose
      if (live) {
        if (kStepChunk) {
          // every trajectory_point_step-th pose for PathAlign (K3); the usual step equals the chunk length: pose 0 of the chunk
          const unsigned k = sample_o + b;
          bufs.samples_x[k] = px[0]; bufs.samples_y[k] = py[0];
          if (sample_yaw) {bufs.samples_yaw[k] = yw[0];}
          sample_o += static_cast<unsigned>(B);
        }
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {
          const int t = t0 + u;
          if (!kTail || t < T) {
            if (!kStepChunk && t == next_sample) {
              const unsigned k = sample_o + b;
              bufs.samples_x[k] = px[u]; bufs.samples_y[k] = py[u];
              if (sample_yaw) {bufs.samples_yaw[k] = yw[u];}
              next_sample += step; sample_o += static_cast<unsigned>(B);
            }
            if (kSpill) {
              const unsigned gu = g + static_cast<unsigned>(u) * static_cast<unsigned>(B);
              if (spill) {bufs.spill_x[gu] = px[u]; bufs.spill_y[gu] = py[u]; bufs.spill_yaw[gu] = yw[u];}
              if (p.vis_b_step > 0 && t % p.vis_t_step == 0 && b % p.vis_b_step == 0) {
                const int nt = (T + p.vis_t_step - 1) / p.vis_t_step;
                const size_t k = static_cast<size_t>(t / p.vis_t_step) * p.vis_nb + b / p.vis_b_step;
                bufs.vis_xy[k] = px[u]; bufs.vis_xy[static_cast<size_t>(nt) * p.vis_nb + k] = py[u];
              }
            }
          }
        }
      }
      g += static_cast<unsigned>(kStreamChunk) * static_cast<unsigned>(B);
      if (kTail) {
#pragma unroll
        for (int u = 0; u < kStreamChunk; ++u) {
          if (t0 + u == T - 1) {ex = px[u]; ey = py[u];}
        }
      } else {
        ex = px[kStreamChunk - 1]; ey = py[kStreamChunk - 1];
      }
      // predict(): state velocities of the next step are the controls of this one (motion_models.hpp:53-66)
      vx = cx[kStreamChunk - 1]; vy = cy[kStreamChunk - 1]; wz = cw[kStreamChunk - 1];
      yaw_prev = yw[kStreamChunk - 1];
    };

  const int T_full = (T / kStreamChunk) * kStreamChunk;
  if (step_is_chunk) {
    for (int t0 = 0; t0 < T_full; t0 += kStreamChunk) {chunk(std::false_type{}, std::true_type{}, t0);}
    if (T_full < T) {chunk(std::true_type{}, std::true_type{}, T_full);}
  } else {
    for (int t0 = 0; t0 < T_full; t0 += kStreamChunk) {chunk(std::false_type{}, std::false_type{}, t0);}
    if (T_full < T) {chunk(std::true_type{}, std::false_type{}, T_full);}
  }

  // furthest reached path point candidate (utils.hpp:292-319): first minimum over the whole path
  unsigned best_j = 0;
  if (p.need_furthest) {
    const float * __restrict__ path_x = reinterpret_cast<const float *>(P + 1) + p.off_path_x;
    const float * __restrict__ path_y = reinterpret_cast<const float *>(P + 1) + p.off_path_y;
    const int N = p.N;
    auto dist2 = [&](int j) {
        const float dx = __fsub_rn(__ldg(path_x + j), ex);
        const float dy = __fsub_rn(__ldg(path_y + j), ey);
        return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
      };
    // The reference scans all N points for the first minimum of the squared distance.  Same answer from a scan that skips:
    // along the path the distance to the end pose cannot fall faster than the path advances, so behind a point at distance
    // r the next floor((r - r_best) / longest segment) points are farther than the best seen so far.  The margins (1e-5
    // relative on both roots; 1 / hmax rounded down by the host) are orders above the rounding of the squared distances
    // (3 fp32 operations) and of sqrt.approx (2^-22), so a skipped point is STRICTLY farther in the kernel's own arithmetic:
    // it can be neither the minimum nor a tie.  A first guess (the point an arc as long as the trajectory's displacement
    // beyond the robot's closest point) makes r_best small from the start; ties go to the lower index as in the reference.
    const float gdx = ex - static_cast<float>(x0), gdy = ey - static_cast<float>(y0);
    const int guess = p.closest_path_pt + __float2int_rn(fminf(sqrt_approx(gdx * gdx + gdy * gdy) * p.path_hmean_inv, 65536.0f));
    best_j = static_cast<unsigned>(max(0, min(N - 1, guess)));
    float best = N > 0 ? dist2(static_cast<int>(best_j)) : 3.402823466e+38f;
    float r_best = sqrt_approx(best);
    const float inv_h = p.path_hmax_inv;
    int j = 0;
    while (j < N) {
      const float d = dist2(j);
      const float r = sqrt_approx(d);
      if (d < best || (d == best && j < static_cast<int>(best_j))) {best = d; best_j = static_cast<unsigned>(j); r_best = r;}
      const float gap = r * 0.99999f - r_best * 1.00001f;
      j += 1 + (gap > 0.0f ? __float2int_rz(fminf(gap * inv_h, 65536.0f)) : 0);
    }
  }

  // publish (same rows as the tile variant)
  const float Tf = static_cast<float>(T);
  float * rows = bufs.crit_rows;
  if (live) {
    bufs.end_xy[b] = ex; bufs.end_xy[B + b] = ey;
    if (con_on) {rows[static_cast<size_t>(p.constraint.idx) * B + b] = add_pow(0.0f, a_con * p.constraint.weight, p.constraint.power);}
    if (fwd_on) {rows[static_cast<size_t>(p.forward.idx) * B + b] = add_pow(0.0f, a_fwd * p.forward.weight, p.forward.power);}
    if (twirl_on) {rows[static_cast<size_t>(p.twirl.idx) * B + b] = add_pow(0.0f, (a_twirl / Tf) * p.twirl.weight, p.twirl.power);}
    if (db_on) {rows[static_cast<size_t>(p.deadband.idx) * B + b] = add_pow(0.0f, a_db * p.deadband.weight, p.deadband.power);}
    if (goal_on) {rows[static_cast<size_t>(p.goal.idx) * B + b] = add_pow(0.0f, (a_goal / Tf) * p.goal.weight, p.goal.power);}
    if (gang_on) {rows[static_cast<size_t>(p.goal_angle.idx) * B + b] = add_pow(0.0f, (a_gang / Tf) * p.goal_angle.weight, p.goal_angle.power);}
    if (cost_on) {
      const float rep = cost_hit ? p.cost_collision : cost_rep;
      rows[static_cast<size_t>(p.cost.idx) * B + b] = add_pow(0.0f, p.cost.weight * rep / Tf, p.cost.power);
    }
    if (ob_on) {
      const float raw = ob_hit ? p.obst_collision : ob_traj;
      const float v = (p.obst_critical_w * raw) + (p.obst_repulsion_w * ob_rep / Tf);
      rows[static_cast<size_t>(p.obst.idx) * B + b] = add_pow(0.0f, v, p.obst.power);
    }
    const size_t gr = static_cast<size_t>(p.n_critics) * B + b;
    rows[gr] = g_vx; rows[gr + B] = g_vy; rows[gr + 2 * static_cast<size_t>(B)] = g_wz;
  }
  if (cost_on) {
    const unsigned ok = __ballot_sync(0xffffffffu, live && !cost_hit);
    if ((tid & 31) == 0 && ok) {atomicOr(&bufs.st->any_ok[p.cost.idx], 1u);}
  }
  if (ob_on) {
    const unsigned ok = __ballot_sync(0xffffffffu, live && !ob_hit);
    if ((tid & 31) == 0 && ok) {atomicOr(&bufs.st->any_ok[p.obst.idx], 1u);}
  }
  if (p.need_furthest) {
    const unsigned m = warp_max_u(live ? best_j : 0u);
    if ((tid & 31) == 0) {atomicMax(&bufs.st->furthest_candidate, m);}
  }
}

// kDevMap: see rollout_score_kernel (the group's batched form takes the member's map pointer from its job instead)
template<unsigned F, bool kExact, bool kDevMap = false>
__global__ void __launch_bounds__(kStreamThreads, MPPI_STREAM_MIN_BLOCKS) rollout_score_stream_kernel(
  const DevParams * __restrict__ P, const uint8_t * __restrict__ cm, DevBuffers bufs)
{
  rollout_score_stream_body<F, kExact>(P, kDevMap ? P->cm_dev : cm, bufs);
}

// ---------------------------------------------------------------------------------------------------
// K3
// ---------------------------------------------------------------------------------------------------
constexpr int kUpdThreads = 128;
constexpr int kMergeT = 4;               // time steps owned by one block of merge_finalize_kernel
constexpr int kLastBlockMergeMax = 64;   // K3's last block merges up to this many partials itself

// utils::findClosestPathPt (utils.hpp:665-675) on the prefix D[0..n); out-of-range clamps to n-1.
// PathAlign calls this with non-decreasing distances, so std::lower_bound over the WHOLE prefix (`cursor`, kept by the
// caller across calls) only ever moves forward: a scan that advances a few entries per call, O(n + calls) per
// trajectory in total.  lower_bound over [init, n) -- what the reference evaluates -- is max(cursor, init).
__device__ __forceinline__ int find_closest_path_pt(const float * D, int n, float dist, int init, int & cursor)
{
  int c = cursor;
  while (c < n && D[c] < dist) {++c;}
  cursor = c;
  const int lo = max(c, init);
  if (lo == init) {return 0;}
  if (lo == n) {return n - 1;}
  if (__fsub_rn(dist, D[lo - 1]) < __fsub_rn(D[lo], dist)) {return lo - 1;}
  return lo;
}

__device__ __forceinline__ void finalize_controls(
  const DevParams * __restrict__ P, const float * __restrict__ merged, float * __restrict__ cs, float * __restrict__ out, int tid, int nthr)
{
  // merged = [min, sum, W_vx[T], W_vy[T], W_wz[T]] ; cs = W / sum, then applyControlSequenceConstraints
  const int T = P->T;
  const float inv = merged[1];
  for (int t = tid; t < T; t += nthr) {
    float vx = merged[2 + t] / inv;
    float wz = merged[2 + 2 * T + t] / inv;
    float vy = cs[T + t];
    if (P->holonomic) {
      vy = merged[2 + T + t] / inv;
      vy = fminf(fmaxf(vy, -P->c_vy), P->c_vy);
    }
    vx = fminf(fmaxf(vx, P->c_vx_min), P->c_vx_max);
    wz = fminf(fmaxf(wz, -P->c_wz), P->c_wz);
    if (P->model == MPPI_MODEL_ACKERMANN) {   // motion_models.hpp:110-117
      const float r = P->min_turning_r;
      if (fabsf(vx) / fabsf(wz) < r) {
        const float sgn = wz > 0.0f ? 1.0f : (wz < 0.0f ? -1.0f : 0.0f);
        wz = sgn * fabsf(vx) / r;
      }
    }
    cs[t] = vx; cs[T + t] = vy; cs[2 * T + t] = wz;
    out[t] = vx; out[T + t] = vy; out[2 * T + t] = wz;
  }
}

// merge n partial records [m, s, W...] (online-softmax merge, SURVEY 8e exchange 2) into dst.
// Called by every thread of one block; `parts` is scratch (slot 0 of each record is overwritten by its scale).
__device__ __forceinline__ void merge_partials(
  float * __restrict__ parts, int n, int stride, int T, float inv_temp, float * dst, float * s_red, int tid, int nthr)
{
  float m = 3.402823466e+38f;
  for (int i = tid; i < n; i += nthr) {m = fminf(m, parts[static_cast<size_t>(i) * stride]);}
  m = warp_min(m);
  if ((tid & 31) == 0) {s_red[tid >> 5] = m;}
  __syncthreads();
  m = s_red[0];
  for (int w = 1; w < nthr / 32; ++w) {m = fminf(m, s_red[w]);}
  __syncthreads();
  for (int i = tid; i < n; i += nthr) {
    float * p = parts + static_cast<size_t>(i) * stride;
    p[0] = expf(-(p[0] - m) * inv_temp);
  }
  __syncthreads();
  for (int c = tid; c < 3 * T + 1; c += nthr) {
    float acc = 0.0f;
#pragma unroll 8
    for (int i = 0; i < n; ++i) {
      const float * p = parts + static_cast<size_t>(i) * stride;
      acc = fmaf(p[1 + c], p[0], acc);
    }
    dst[1 + c] = acc;
  }
  if (tid == 0) {dst[0] = m;}
}

// The scalar decisions of one CriticManager::evalTrajectoriesScores pass (critic_manager.cpp:67-76), taken once per
// block by one thread: which critic raised fail_flag, the furthest reached path point, and the path critics' gates.
struct K3Decisions
{
  int fail_at;        // index of the critic that raised fail_flag (critics after it are skipped); n_critics if none
  int furthest, furthest_set;
  int follow_idx;
  int align_go, legacy_go, angle_go, angle_idx;
};

// shared-memory carve-up common to the K3 kernels: hot | D[N] | path x[N] | path y[N] | valid[N] | flags[N] | follow_idx[N]
__host__ __device__ inline size_t k3_common_smem_bytes()
{
  return kHotBytes + 3 * sizeof(float) * MPPI_MAX_PATH_POINTS + 2 * MPPI_MAX_PATH_POINTS + sizeof(uint16_t) * (MPPI_MAX_PATH_POINTS + 16);
}

struct K3Path
{
  const float * x, * y, * yaw;     // global (read through the read-only path)
  const float * s_D;               // shared: arc-length prefix
  const float * s_x, * s_y;        // shared copies of the path points (PathAlign's data-dependent look-ups)
  const uint8_t * s_valid;         // shared: path point validity (utils::findPathCosts, host decided)
};

// The decisions themselves (one thread).  any_ok / state = {furthest_candidate, furthest, furthest_set, fail_flag} are this
// pass's reductions over all trajectories (after exchange 1 when sharded); flags / follow are the host-made tables indexed
// by the furthest reached path point (build_params).
__device__ __forceinline__ void k3_decide(
  const DevParams * P, int N, const unsigned * any_ok, const unsigned * state, const uint8_t * s_flags, const uint16_t * s_follow,
  int iteration, K3Decisions * dec)
{
  const int nc = P->n_critics;
  // CriticManager::evalTrajectoriesScores (critic_manager.cpp:67-76): the first obstacle-type critic (list order)
  // that saw no surviving trajectory raises fail_flag; critics after it are skipped
  int fail_at = nc;
  if (iteration > 0 && state[3]) {
    fail_at = -1;     // fail_flag is only cleared in prepare(): a failed iteration mutes the following ones
  } else {
    const int q0 = P->obstacle_q[0], q1 = P->obstacle_q[1];
    if (q0 >= 0 && any_ok[q0] == 0u) {
      fail_at = q0;
    } else if (q1 >= 0 && any_ok[q1] == 0u) {
      fail_at = q1;
    }
  }
  unsigned furthest;
  int fset;
  if (iteration == 0) {
    fset = P->preset_furthest != kUnset; furthest = fset ? P->preset_furthest : 0u;
  } else {
    fset = static_cast<int>(state[2]); furthest = state[1];
  }
  // the first enabled path critic in list order calls setPathFurthestPointIfNotSet (utils.hpp:350-355)
  if (!fset && P->first_path_q >= 0 && P->first_path_q <= fail_at) {furthest = state[0]; fset = 1;}
  const int f = min(static_cast<int>(furthest), N - 1);
  const unsigned flags = s_flags[f];
  dec->fail_at = fail_at;
  dec->furthest = static_cast<int>(furthest);
  dec->furthest_set = fset;
  dec->follow_idx = (P->follow.on && P->follow.idx <= fail_at) ? s_follow[f] : 0;
  dec->align_go = (P->align.on && P->align.idx <= fail_at && (flags & 1u)) ? 1 : 0;
  dec->legacy_go = (P->legacy.on && P->legacy.idx <= fail_at && (flags & 2u)) ? 1 : 0;
  dec->angle_go = (P->angle.on && P->angle.idx <= fail_at && (flags & 4u)) ? 1 : 0;
  dec->angle_idx = min(static_cast<int>(furthest) + P->angle_offset, N - 1);
}

// Copies the hot record, the path and its host-made tables into shared memory and lets thread 0 take the decisions.
// Memory round trips are the cost here (a cold record is ~1 us away), so everything is requested in one wave.  The
// decisions that depend on device results (which critic failed, the furthest reached point) are a handful of
// table look-ups: everything that is a function of "furthest" alone was tabulated by the host (build_params).
__device__ __forceinline__ void k3_preamble(
  float * smem, const DevParams * __restrict__ Pg, DevState * st, const PeerComm & pc, int iteration, int tid, int nthr, K3Path & path,
  K3Decisions * dec)
{
  __shared__ unsigned s_any_ok[kMaxCritics];
  __shared__ unsigned s_state[4];   // furthest_candidate, furthest, furthest_set, fail_flag
  float * s_hot = smem;
  const int N = Pg->N;              // read straight from the record: the path copies need not wait for the barrier
  load_hot_params(s_hot, Pg, tid, nthr);
  const DevParams * P = reinterpret_cast<const DevParams *>(s_hot);
  const float * tail = reinterpret_cast<const float *>(Pg + 1);
  // record tail layout (build_params): x[N] y[N] yaw[N] D[N] | valid[n16] flags[n16] follow_idx[N] (uint16)
  const int n16 = ((N + 15) / 16) * 16;
  path.x = tail; path.y = tail + N; path.yaw = tail + 2 * N;
  const uint8_t * g_valid = reinterpret_cast<const uint8_t *>(tail + 4 * N);
  const uint8_t * g_flags = g_valid + n16;
  const uint16_t * g_follow = reinterpret_cast<const uint16_t *>(g_valid + 2 * n16);
  float * s_D = s_hot + kHotFloats;
  float * s_px = s_D + MPPI_MAX_PATH_POINTS, * s_py = s_px + MPPI_MAX_PATH_POINTS;
  uint8_t * s_valid = reinterpret_cast<uint8_t *>(s_py + MPPI_MAX_PATH_POINTS);
  uint8_t * s_flags = s_valid + MPPI_MAX_PATH_POINTS;
  uint16_t * s_follow = reinterpret_cast<uint16_t *>(s_flags + MPPI_MAX_PATH_POINTS);
  path.s_D = s_D; path.s_x = s_px; path.s_y = s_py; path.s_valid = s_valid;
  {
    const float * g_D = tail + 3 * N;
    for (int j = tid; j < N; j += nthr) {
      s_D[j] = __ldg(g_D + j); s_px[j] = __ldg(path.x + j); s_py[j] = __ldg(path.y + j);
      s_valid[j] = __ldg(g_valid + j); s_flags[j] = __ldg(g_flags + j); s_follow[j] = __ldg(g_follow + j);
    }
  }
  // everything above is the cycle's upload (complete before the rollout kernel started); what follows reads the rollout
  // kernel's reductions: under a programmatic dependent launch this is where the block waits for it
  pdl_wait();
  if (tid < kMaxCritics) {s_any_ok[tid] = st->any_ok[tid];}
  if (tid == 32) {s_state[0] = st->furthest_candidate; s_state[1] = st->furthest;}
  if (tid == 33) {s_state[2] = static_cast<unsigned>(st->furthest_set); s_state[3] = static_cast<unsigned>(st->fail_flag);}
  if (pc.nranks > 1) {
    // ---- exchange 1 over peer memory: element-wise MAX of (furthest candidate, survivor flags) across the ranks.
    //      Block 0 pushes this rank's 17 words as packets into every mailbox; every block polls its LOCAL mailbox.
    __shared__ unsigned s_x1[1 + kMaxCritics];
    const unsigned tag = ld_volatile_u32(pc.seq) + 1u;
    constexpr int kWords = 1 + kMaxCritics;
    if (tid < kWords) {s_x1[tid] = 0u;}
    if (blockIdx.x == 0 && tid < kWords) {
      const unsigned v = tid == 0 ? st->furthest_candidate : st->any_ok[tid - 1];
#pragma unroll 1
      for (int r = 0; r < pc.nranks; ++r) {st_packet(pc.box[r] + kBoxX1 + pc.rank * kX1Words + tid, v, tag);}
    }
    __syncthreads();
    const uint2 * local = pc.box[pc.rank];
    for (int i = tid; i < kWords * pc.nranks; i += nthr) {
      const int r = i / kWords, w = i - r * kWords;
      unsigned v;
      if (!poll_packet(local + kBoxX1 + r * kX1Words + w, tag, v)) {st->comm_error = 1u;}
      atomicMax(&s_x1[w], v);
    }
    __syncthreads();
    if (tid < kWords) {
      if (tid == 0) {s_state[0] = s_x1[0];} else {s_any_ok[tid - 1] = s_x1[tid];}
    }
  }
  MPPI_TRACE_AT(24);
  __syncthreads();
  MPPI_TRACE_AT(25);
  if (tid == 0) {k3_decide(P, N, s_any_ok, s_state, s_flags, s_follow, iteration, dec);}
  MPPI_TRACE_AT(26);
  __syncthreads();
}

// One trajectory: the path critics, then the total in critic-list order (fail_flag short-circuit) and the gamma term.
__device__ __forceinline__ float k3_trajectory_total(
  int b, const DevParams * P, const K3Decisions & dec, const K3Path & path, const DevBuffers & bufs, int iteration)
{
  const int T = P->T, B = P->B, N = P->N, nc = P->n_critics;
  const int fail_at = dec.fail_at, furthest = dec.furthest;
  const float * s_D = path.s_D;
  const uint8_t * s_valid = path.s_valid;
  const float * __restrict__ path_x = path.x;
  const float * __restrict__ path_y = path.y;
  const float * __restrict__ path_yaw = path.yaw;
  float total = (iteration == 0 && P->mode == 0) ? 0.0f : bufs.costs[b];
  float * rows = bufs.crit_rows;
  // every K2 row this trajectory will need, requested up front: one memory round trip instead of one per critic
  float row_v[kMaxCritics];
#pragma unroll
  for (int q = 0; q < kMaxCritics; ++q) {
    row_v[q] = 0.0f;
    if (q < nc && q <= fail_at) {
      const int kind = P->kind_of[q];
      const bool from_k3 = kind == MPPI_CRITIC_PATH_FOLLOW || kind == MPPI_CRITIC_PATH_ALIGN ||
        kind == MPPI_CRITIC_PATH_ALIGN_LEGACY || kind == MPPI_CRITIC_PATH_ANGLE;
      if (!from_k3) {row_v[q] = rows[static_cast<size_t>(q) * B + b];}
    }
  }
  float gam[3] = {0.0f, 0.0f, 0.0f};
  if (P->mode == 0) {
    const size_t g = static_cast<size_t>(nc) * B + b;
    gam[0] = rows[g]; gam[1] = rows[g + B]; gam[2] = rows[g + 2 * static_cast<size_t>(B)];
  }
  const float end_x = bufs.end_xy[b], end_y = bufs.end_xy[B + b];
  for (int q = 0; q < nc; ++q) {
    if (q > fail_at) {break;}
    const int kind = P->kind_of[q];
    float term = 0.0f;
    bool has = false;
    switch (kind) {
      case MPPI_CRITIC_PATH_FOLLOW:
        if (P->follow.on) {    // path_follow_critic.cpp:60-70
          const float dx = end_x - path.s_x[dec.follow_idx];
          const float dy = end_y - path.s_y[dec.follow_idx];
          term = add_pow(0.0f, P->follow.weight * sqrtf(dx * dx + dy * dy), P->follow.power);
          has = true;
        }
        break;
      case MPPI_CRITIC_PATH_ALIGN:
        if (dec.align_go) {     // path_align_critic.cpp:92-135, sequential and in the reference's fp32 order
          const int step = P->align_step;
          const int n_s = (T + step - 1) / step;     // sampled poses p = 0, step, 2 step, ... < T
          float traj_d = 0.0f, summed = 0.0f, num = 0.0f;
          int path_pt = 0, cursor = 0;
          float prev_x = bufs.samples_x[b], prev_y = bufs.samples_y[b];
          constexpr int kBatch = 8;                  // sampled poses requested together (latency off the serial chain)
          for (int k0 = 1; k0 < n_s; k0 += kBatch) {
            float sx[kBatch], sy[kBatch], syaw[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
              const int k = min(k0 + u, n_s - 1);
              sx[u] = bufs.samples_x[static_cast<size_t>(k) * B + b];
              sy[u] = bufs.samples_y[static_cast<size_t>(k) * B + b];
              syaw[u] = P->align_use_yaw ? bufs.samples_yaw[static_cast<size_t>(k) * B + b] : 0.0f;
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
              if (k0 + u < n_s) {
                const float Tx = sx[u], Ty = sy[u];
                float dx = __fsub_rn(Tx, prev_x), dy = __fsub_rn(Ty, prev_y);
                traj_d = __fadd_rn(traj_d, __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))));
                path_pt = find_closest_path_pt(s_D, furthest, traj_d, path_pt, cursor);
                if (s_valid[path_pt]) {
                  dx = __fsub_rn(path.s_x[path_pt], Tx);
                  dy = __fsub_rn(path.s_y[path_pt], Ty);
                  num = __fadd_rn(num, 1.0f);
                  // the distance itself only feeds the cost (1e-4 tolerance): one MUFU instead of the IEEE sequence
                  if (P->align_use_yaw) {
                    const float dyaw = static_cast<float>(normalize_angle_d(static_cast<double>(syaw[u]) - static_cast<double>(__ldg(path_yaw + path_pt))));
                    summed += sqrt_approx(dx * dx + dy * dy + dyaw * dyaw);
                  } else {
                    summed += sqrt_approx(dx * dx + dy * dy);
                  }
                }
                prev_x = Tx; prev_y = Ty;
              }
            }
          }
          const float cost = num > 0.0f ? __fdiv_rn(summed, num) : 0.0f;
          term = add_pow(0.0f, __fmul_rn(cost, P->align.weight), P->align.power);
          has = true;
        }
        break;
      case MPPI_CRITIC_PATH_ALIGN_LEGACY:
        if (dec.legacy_go) {    // path_align_legacy_critic.cpp:97-128
          const int step = P->legacy_step;
          const int segs = N - 1;
          float summed = 0.0f;
          int k = 1;
          for (int p = step; p < T; p += step, ++k) {
            const float Tx = bufs.samples_x[static_cast<size_t>(k) * B + b];
            const float Ty = bufs.samples_y[static_cast<size_t>(k) * B + b];
            float Tyaw = 0.0f;
            if (P->legacy_use_yaw) {Tyaw = bufs.samples_yaw[static_cast<size_t>(k) * B + b];}
            float min_d = 3.402823466e+38f;
            int min_s = 0;
            for (int sgm = 0; sgm < segs - 1; ++sgm) {
              const float dx = __fsub_rn(__ldg(path_x + sgm), Tx);
              const float dy = __fsub_rn(__ldg(path_y + sgm), Ty);
              float d = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
              if (P->legacy_use_yaw) {
                const float dyaw = static_cast<float>(normalize_angle_d(static_cast<double>(Tyaw) - static_cast<double>(__ldg(path_yaw + sgm))));
                d = __fadd_rn(d, __fmul_rn(dyaw, dyaw));
              }
              if (d < min_d) {min_d = d; min_s = sgm;}
            }
            if (min_s != 0 && s_valid[min_s]) {summed = __fadd_rn(summed, __fsqrt_rn(min_d));}
          }
          const float evals = static_cast<float>(T / step);
          term = add_pow(0.0f, __fmul_rn(__fdiv_rn(summed, evals), P->legacy.weight), P->legacy.power);
          has = true;
        }
        break;
      case MPPI_CRITIC_PATH_ANGLE:
        if (dec.angle_go) {     // path_angle_critic.cpp:85-100
          const float gx = __ldg(path_x + dec.angle_idx), gy = __ldg(path_y + dec.angle_idx);
          float sum = 0.0f;
          for (int t = 0; t < T; ++t) {
            const size_t g = static_cast<size_t>(t) * B + b;
            const float x = bufs.spill_x[g], y = bufs.spill_y[g], yaw = bufs.spill_yaw[g];
            const float ybp = atan2f(__fsub_rn(gy, y), __fsub_rn(gx, x));
            double v = fabs(normalize_angle_d(static_cast<double>(__fsub_rn(ybp, yaw))));
            if (P->angle_reversing && !P->angle_forward_pref) {
              const double corrected = v < 1.57079632679489661923 ? static_cast<double>(ybp) :
                normalize_angle_d(static_cast<double>(ybp) + 3.14159265358979323846);
              v = fabs(normalize_angle_d(corrected - static_cast<double>(yaw)));
            }
            sum += static_cast<float>(v);
          }
          term = add_pow(0.0f, (sum / static_cast<float>(T)) * P->angle.weight, P->angle.power);
          has = true;
        }
        break;
      case MPPI_CRITIC_CONSTRAINT: has = P->constraint.on; break;
      case MPPI_CRITIC_COST: has = P->cost.on; break;
      case MPPI_CRITIC_GOAL: has = P->goal.on; break;
      case MPPI_CRITIC_GOAL_ANGLE: has = P->goal_angle.on; break;
      case MPPI_CRITIC_OBSTACLES: has = P->obst.on; break;
      case MPPI_CRITIC_PREFER_FORWARD: has = P->forward.on; break;
      case MPPI_CRITIC_TWIRLING: has = P->twirl.on; break;
      case MPPI_CRITIC_VELOCITY_DEADBAND: has = P->deadband.on; break;
      default: break;
    }
    const bool from_k3 = kind == MPPI_CRITIC_PATH_FOLLOW || kind == MPPI_CRITIC_PATH_ALIGN ||
      kind == MPPI_CRITIC_PATH_ALIGN_LEGACY || kind == MPPI_CRITIC_PATH_ANGLE;
    if (from_k3) {
      if (P->want_critic_rows) {rows[static_cast<size_t>(q) * B + b] = term;}   // for the per-critic getter
    } else if (has) {
#pragma unroll
      for (int r = 0; r < kMaxCritics; ++r) {term = r == q ? row_v[r] : term;}   // register array: static indices only
    }
    if (has) {total = __fadd_rn(total, term);}
  }
  if (P->want_critic_rows) {
    // rows of critics that did not run read as zero for the per-critic getter (mppi_get_critic_costs)
    for (int q = 0; q < nc; ++q) {
      const int kind = P->kind_of[q];
      const bool from_k3 = kind == MPPI_CRITIC_PATH_FOLLOW || kind == MPPI_CRITIC_PATH_ALIGN ||
        kind == MPPI_CRITIC_PATH_ALIGN_LEGACY || kind == MPPI_CRITIC_PATH_ANGLE;
      bool on = false;
      switch (kind) {
        case MPPI_CRITIC_CONSTRAINT: on = P->constraint.on; break;
        case MPPI_CRITIC_COST: on = P->cost.on; break;
        case MPPI_CRITIC_GOAL: on = P->goal.on; break;
        case MPPI_CRITIC_GOAL_ANGLE: on = P->goal_angle.on; break;
        case MPPI_CRITIC_OBSTACLES: on = P->obst.on; break;
        case MPPI_CRITIC_PREFER_FORWARD: on = P->forward.on; break;
        case MPPI_CRITIC_TWIRLING: on = P->twirl.on; break;
        case MPPI_CRITIC_VELOCITY_DEADBAND: on = P->deadband.on; break;
        default: break;
      }
      if (q > fail_at || (!from_k3 && !on)) {rows[static_cast<size_t>(q) * B + b] = 0.0f;}
    }
  }
  if (P->mode == 0) {
    // gamma term (optimizer.cpp:367-380): vx, then wz, then vy (holonomic)
    total = __fadd_rn(total, __fmul_rn(P->gamma_vx, gam[0]));
    total = __fadd_rn(total, __fmul_rn(P->gamma_wz, gam[2]));
    if (P->holonomic) {total = __fadd_rn(total, __fmul_rn(P->gamma_vy, gam[1]));}
  }
  bufs.costs[b] = total;
  return total;
}

// out-of-line instance for path_costs_tm_body: the general total must not cost the lean one beside it registers
__device__ __noinline__ float k3_trajectory_total_general(
  int b, const DevParams * P, const K3Decisions & dec, const K3Path & path, const DevBuffers & bufs, int iteration)
{
  return k3_trajectory_total(b, P, dec, path, bufs, iteration);
}

// The same total for the usual case, at 60 % of the instructions: no per-critic rows requested, PathAlign without path
// orientations, PathAlignLegacy / PathAngle not firing this pass (block-uniform conditions, decided once per block in
// path_costs_tm_body).  `src` = where the term of list position q comes from this pass, one byte per position
// (0 nothing, 1 K2's row, 2 PathFollow, 3 PathAlign), packed four to a word so that the unrolled loops index registers
// statically.  PathAlign (path_align_critic.cpp:92-135): utils::findClosestPathPt's lower_bound (utils.hpp:665-675) is a
// cursor that only moves forward from sample to sample, placed by a guess from the path's mean spacing (`inv_h`, points
// per metre) and corrected both ways against the arc-length table; the answer follows from the cursor and the previous
// answer by selects.  The tables are read by 32-bit shared-window addresses (lds_f32).
__device__ __forceinline__ float k3_trajectory_total_fast(
  int b, const DevParams * P, const K3Decisions & dec, const K3Path & path, const DevBuffers & bufs, int iteration, const unsigned (&src_w)[kMaxCritics / 4], const float inv_h)
{
  const int T = P->T, B = P->B;
  const float * __restrict__ rows = bufs.crit_rows;
  float row_v[kMaxCritics];
#pragma unroll
  for (int q = 0; q < kMaxCritics; ++q) {
    const unsigned src = (src_w[q >> 2] >> (8 * (q & 3))) & 0xffu;
    row_v[q] = src == 1u ? rows[static_cast<size_t>(q) * B + b] : 0.0f;
  }
  float total = iteration == 0 ? 0.0f : bufs.costs[b];
  const size_t g = static_cast<size_t>(P->n_critics) * B + b;
  const float gam0 = rows[g], gam1 = rows[g + B], gam2 = rows[g + 2 * static_cast<size_t>(B)];
  float follow_term = 0.0f, align_term = 0.0f;
  if (P->follow.on) {    // path_follow_critic.cpp:60-70
    const float dx = bufs.end_xy[b] - path.s_x[dec.follow_idx];
    const float dy = bufs.end_xy[B + b] - path.s_y[dec.follow_idx];
    follow_term = add_pow(0.0f, P->follow.weight * sqrtf(dx * dx + dy * dy), P->follow.power);
  }
  if (dec.align_go) {
    const int n = dec.furthest;
    const int step = P->align_step;
    const int n_s = (T + step - 1) / step;     // sampled poses p = 0, step, 2 step, ... < T
    const float * __restrict__ sxp = bufs.samples_x + b;
    const float * __restrict__ syp = bufs.samples_y + b;
    // the path tables by shared-window address: D[j] at aD + 4 j, x[j] / y[j] one / two table pitches behind it, valid[j]
    // at aV + j (k3_preamble's carve-up)
    const unsigned aD = smem_addr(path.s_D), aV = smem_addr(path.s_valid);
    constexpr unsigned kPitch = 4u * MPPI_MAX_PATH_POINTS;
    const unsigned a_end = aD + 4u * static_cast<unsigned>(n), a_last = aD + 4u * static_cast<unsigned>(max(n - 1, 0));
    unsigned a_c = aD;                         // address of D[c], c = lower_bound(D[0, n), distance): only ever moves forward
    unsigned a_prev = aD;                      // address of D[previous answer]
    float traj_d = 0.0f, summed = 0.0f, num = 0.0f;
    float prev_x = sxp[0], prev_y = syp[0];
    const float kInf = __int_as_float(0x7f800000);
    auto sample = [&](const float Tx, const float Ty) {
        const float ddx = __fsub_rn(Tx, prev_x), ddy = __fsub_rn(Ty, prev_y);
        traj_d = __fadd_rn(traj_d, __fsqrt_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy))));
        // lower_bound by a guess from the mean spacing of the path (exact for an evenly spaced path up to rounding), then
        // corrected both ways against the table itself: D[c - 1] < distance <= D[c].  Any guess gives the same c; the two
        // table entries that prove it are the ones the nearest-neighbour decision needs.
        const unsigned a_g = aD + 4u * static_cast<unsigned>(__float2int_rd(__fmul_rn(traj_d, inv_h)) + 1);
        const unsigned a_0 = a_c;              // lower_bound is monotone in the distance: never below the previous cursor
        a_c = min(max(a_g, a_0), a_end);
        float d_lo = a_c < a_end ? lds_f32(a_c) : kInf;                           // D[c]     (+inf at the end of the prefix)
        float d_lm = a_c > aD ? lds_f32(a_c - 4u) : -kInf;                        // D[c - 1] (-inf in front of it)
        while (d_lo < traj_d) {
          a_c += 4u; d_lm = d_lo;
          d_lo = a_c < a_end ? lds_f32(a_c) : kInf;
        }
        while (a_c > a_0 && d_lm >= traj_d) {
          a_c -= 4u; d_lo = d_lm;
          d_lm = a_c > aD ? lds_f32(a_c - 4u) : -kInf;
        }
        // findClosestPathPt over [init, n), init = the previous answer: 0 when the bound does not pass init, the last
        // point when it runs off the prefix, else the nearer of the two neighbours
        const unsigned a_near = __fsub_rn(traj_d, d_lm) < __fsub_rn(d_lo, traj_d) ? a_c - 4u : a_c;
        const unsigned a_res = a_c <= a_prev ? aD : (a_c == a_end ? a_last : a_near);
        a_prev = a_res;
        const float ex = __fsub_rn(lds_f32(a_res + kPitch), Tx), ey = __fsub_rn(lds_f32(a_res + 2u * kPitch), Ty);
        if (lds_u8(aV + ((a_res - aD) >> 2))) {
          num = __fadd_rn(num, 1.0f);
          // the distance itself only feeds the cost (1e-4 tolerance): one MUFU instead of the IEEE sequence
          summed += sqrt_approx(ex * ex + ey * ey);
        }
        prev_x = Tx; prev_y = Ty;
      };
    constexpr int kBatch = 8;                  // sampled poses requested together (latency off the serial chain)
    int k0 = 1;
    unsigned o = static_cast<unsigned>(B);
    for (; k0 + kBatch <= n_s; k0 += kBatch) {
      float sx[kBatch], sy[kBatch];
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {sx[u] = sxp[o]; sy[u] = syp[o]; o += static_cast<unsigned>(B);}
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {sample(sx[u], sy[u]);}
    }
    for (; k0 < n_s; ++k0) {
      const float Tx = sxp[o], Ty = syp[o];
      o += static_cast<unsigned>(B);
      sample(Tx, Ty);
    }
    const float cost = num > 0.0f ? __fdiv_rn(summed, num) : 0.0f;
    align_term = add_pow(0.0f, __fmul_rn(cost, P->align.weight), P->align.power);
  }
#pragma unroll
  for (int q = 0; q < kMaxCritics; ++q) {
    const unsigned src = (src_w[q >> 2] >> (8 * (q & 3))) & 0xffu;
    if (src != 0u) {
      const float term = src == 1u ? row_v[q] : (src == 2u ? follow_term : align_term);
      total = __fadd_rn(total, term);
    }
  }
  // gamma term (optimizer.cpp:367-380): vx, then wz, then vy (holonomic)
  total = __fadd_rn(total, __fmul_rn(P->gamma_vx, gam0));
  total = __fadd_rn(total, __fmul_rn(P->gamma_wz, gam2));
  if (P->holonomic) {total = __fadd_rn(total, __fmul_rn(P->gamma_vy, gam1));}
  bufs.costs[b] = total;
  return total;
}

// flags of the pass, published by the last block to finish
__device__ __forceinline__ void k3_publish_flags(const DevParams * P, DevState * st, const K3Decisions & dec, float * out)
{
  const int T = P->T;
  st->fail_flag = dec.fail_at < P->n_critics ? 1 : 0;
  st->furthest = static_cast<unsigned>(dec.furthest);
  st->furthest_set = dec.furthest_set;
  st->furthest_candidate = 0u;
  for (int q = 0; q < kMaxCritics; ++q) {st->any_ok[q] = 0u;}
  st->ticket = 0u;
  out[3 * T] = __int_as_float(st->fail_flag);
  out[3 * T + 1] = __uint_as_float(dec.furthest_set ? static_cast<unsigned>(dec.furthest) : kUnset);
}

// K3, stream layout: path critics + totals for every trajectory (grid-stride: the preamble is paid once per block,
// not once per 128 trajectories) and the global minimum of the costs; the weighted sums follow in
// weighted_sums_tm_kernel.
// kMinBlocks trades registers for occupancy: 8 resident blocks (64 registers, a few spills) win once the batch keeps every
// SM oversubscribed, 5 (96 registers) below that (measured on B200, profiles/).
// bump_epoch: the last block also advances the handle's packet epoch, so that the merge kernel behind this one can tag the
// result packets it writes to pinned host memory (stream layout, unsharded: no copy node, no stream synchronisation)
// nblocks: the blocks that work on this problem (blockIdx.x < nblocks), i.e. its grid stride, ticket count and number of
// partial minima; gridDim.x for one handle, the member's own count in a group launched at the largest member's extent
__device__ __forceinline__ void path_costs_tm_body(const DevParams * __restrict__ Pg, const DevBuffers & bufs, int iteration, int bump_epoch,
  unsigned nblocks)
{
  extern __shared__ float smem[];
  __shared__ K3Decisions dec;
  __shared__ float s_red[kUpdThreads / 32];
  __shared__ unsigned sc_last;
  const int tid = threadIdx.x;
  pdl_launch_dependents();   // the weighted-sums kernel may set up its ring and request its first noise rows meanwhile
  K3Path path;
  k3_preamble(smem, Pg, bufs.st, bufs.peer, iteration, tid, kUpdThreads, path, &dec);
  const DevParams * P = reinterpret_cast<const DevParams *>(smem);
  const int B = P->B, T = P->T;
  float m = 3.402823466e+38f;
  // block-uniform: the usual pass runs the lean total (k3_trajectory_total_fast), anything else the general one
  const bool fast = P->mode == 0 && !P->want_critic_rows && !dec.legacy_go && !dec.angle_go && !(dec.align_go && P->align_use_yaw);
  __shared__ unsigned s_srcw[kMaxCritics / 4];
  if (tid < kMaxCritics / 4) {   // where the term of every list position comes from this pass, four positions to a word
    unsigned v = 0u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int q = 4 * tid + i;
      unsigned src = (q < P->n_critics && q <= dec.fail_at) ? P->src_base[q] : 0u;
      if ((src == 3u && !dec.align_go) || src >= 4u) {src = 0u;}
      v |= src << (8 * i);
    }
    s_srcw[tid] = v;
  }
  __syncthreads();
  if (fast) {
    unsigned src_w[kMaxCritics / 4];
#pragma unroll
    for (int w = 0; w < kMaxCritics / 4; ++w) {src_w[w] = s_srcw[w];}
    // points per metre of the path: the start of the per-sample search in the arc-length prefix (efficiency only)
    const float d_all = path.s_D[max(P->N - 1, 0)];
    const float inv_h = d_all > 0.0f ? static_cast<float>(P->N - 1) / d_all : 0.0f;
    for (int base = blockIdx.x * kUpdThreads; base < B; base += nblocks * kUpdThreads) {
      const int b = base + tid;
      if (b < B) {m = fminf(m, k3_trajectory_total_fast(b, P, dec, path, bufs, iteration, src_w, inv_h));}
    }
  } else {
    for (int base = blockIdx.x * kUpdThreads; base < B; base += nblocks * kUpdThreads) {
      const int b = base + tid;
      if (b < B) {m = fminf(m, k3_trajectory_total_general(b, P, dec, path, bufs, iteration));}
    }
  }
  m = warp_min(m);
  if ((tid & 31) == 0) {s_red[tid >> 5] = m;}
  __syncthreads();
  const int stride = 3 * T + 2;
  if (tid == 0) {
#pragma unroll
    for (int w = 1; w < kUpdThreads / 32; ++w) {m = fminf(m, s_red[w]);}
    bufs.partials[static_cast<size_t>(blockIdx.x) * stride] = m;
    __threadfence();
    sc_last = atomicAdd(&bufs.st->ticket, 1u) == nblocks - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (!sc_last) {return;}
  __threadfence();
  float gm = 3.402823466e+38f;
  for (int i = tid; i < static_cast<int>(nblocks); i += kUpdThreads) {gm = fminf(gm, bufs.partials[static_cast<size_t>(i) * stride]);}
  gm = warp_min(gm);
  __syncthreads();
  if ((tid & 31) == 0) {s_red[tid >> 5] = gm;}
  __syncthreads();
  if (tid == 0) {
    gm = s_red[0];
    for (int w = 1; w < kUpdThreads / 32; ++w) {gm = fminf(gm, s_red[w]);}
    bufs.st->global_min = gm;
    k3_publish_flags(P, bufs.st, dec, bufs.out);
    if (bump_epoch) {*bufs.epoch += 1u;}
  }
}

template<int kMinBlocks>
__global__ void __launch_bounds__(kUpdThreads, kMinBlocks) path_costs_tm_kernel(
  const DevParams * __restrict__ Pg, const __grid_constant__ DevBuffers bufs, int iteration, int bump_epoch)
{
  path_costs_tm_body(Pg, bufs, iteration, bump_epoch, gridDim.x);
}

// K3, tile layout (small and medium batches; latency matters more than throughput here).  One block owns
// kUpdRows = 32 trajectories.  Warp 0 walks the per-trajectory critic totals (one lane per trajectory) while the
// other warps stage the block's noise rows [32][3][T] into shared memory, so the weighted column sums that follow
// the softmax run out of shared memory with all threads busy.  The last block to finish merges the per-block
// online-softmax records and writes the new control sequence (up to kLastBlockMergeMax blocks; beyond that
// merge_finalize_kernel does it in parallel).
constexpr int kUpdRows = 32;
__host__ __device__ inline size_t k3_tile_smem_bytes(int T)
{
  return k3_common_smem_bytes() + sizeof(float) * (static_cast<size_t>(kUpdRows) * 3 * T + kUpdRows + 8);
}

__global__ void __launch_bounds__(kUpdThreads) path_softmax_update_kernel(
  const DevParams * __restrict__ Pg, DevBuffers bufs, int n_ranks, int iteration, const int B0, const int T0, const int mode0)
{
  extern __shared__ float smem[];
  __shared__ K3Decisions dec;
  __shared__ unsigned sc_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  MPPI_TRACE_AT(16);
  // the noise rows do not depend on anything K3 decides: request them before the preamble's barriers
  // (B0, T0, mode0 repeat the record's B, T, mode as launch arguments: no memory round trip before the first load)
  float * s_tile = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(smem) + k3_common_smem_bytes());   // [32][3T]
  float * s_w = s_tile + static_cast<size_t>(kUpdRows) * 3 * T0;                                             // [32]
  float * s_stat = s_w + kUpdRows;                                                                           // [m, ssum]
  const int rows_here = min(kUpdRows, B0 - static_cast<int>(blockIdx.x) * kUpdRows);
  if (mode0 == 0 && warp > 0) {
    const int nstage = kUpdThreads - 32, sid = tid - 32;
    const size_t row0 = static_cast<size_t>(blockIdx.x) * kUpdRows * T0;
    if ((T0 & 3) == 0) {
      const int rs = T0 >> 2, per_plane = rows_here * rs;
      for (int i = sid; i < 3 * per_plane; i += nstage) {
        const int plane = i / per_plane, j = i - plane * per_plane;
        const int r = j / rs, q4 = j - r * rs;
        const float * src = (plane == 0 ? bufs.in_a : (plane == 1 ? bufs.in_b : bufs.in_c)) + row0;
        const float4 v = __ldg(reinterpret_cast<const float4 *>(src) + j);
        *reinterpret_cast<float4 *>(s_tile + (static_cast<size_t>(r) * 3 + plane) * T0 + 4 * q4) = v;
      }
    } else {
      const int per_plane = rows_here * T0;
      for (int i = sid; i < 3 * per_plane; i += nstage) {
        const int plane = i / per_plane, j = i - plane * per_plane;
        const int r = j / T0, t = j - r * T0;
        const float * src = (plane == 0 ? bufs.in_a : (plane == 1 ? bufs.in_b : bufs.in_c)) + row0;
        s_tile[(static_cast<size_t>(r) * 3 + plane) * T0 + t] = __ldg(src + j);
      }
    }
  }
  MPPI_TRACE_AT(17);
  K3Path path;
  k3_preamble(smem, Pg, bufs.st, bufs.peer, iteration, tid, kUpdThreads, path, &dec);
  const DevParams * P = reinterpret_cast<const DevParams *>(smem);   // hot fields only; arrays stay in global (Pg)
  const int T = P->T, B = P->B;
  DevState * st = bufs.st;

  MPPI_TRACE_AT(18);
  // ---- phase 1: warp 0, one lane per trajectory: path critics + total in list order; block-local softmax record
  const float inv_temp = 1.0f / P->temperature;
  if (warp == 0) {
    const int b = blockIdx.x * kUpdRows + lane;
    const bool live = b < B;
    float total = 3.402823466e+38f;
    if (live) {total = k3_trajectory_total(b, P, dec, path, bufs, iteration);}
    if (P->mode == 0) {
      // optimizer.cpp:382-391 on this block's rows: m = min, w = exp(-(c - m) / temperature), s = sum w
      const float m = warp_min(total);
      const float w_b = live ? expf(-(total - m) * inv_temp) : 0.0f;
      const float ssum = warp_sum(w_b);
      s_w[lane] = w_b;
      if (lane == 0) {s_stat[0] = m; s_stat[1] = ssum;}
    }
  }
  MPPI_TRACE_AT(19);
  if (P->mode != 0) {
    // score mode: no control update; the last block publishes the flags
    __threadfence();
    __syncthreads();
    if (tid == 0) {sc_last = atomicAdd(&st->ticket, 1u) == gridDim.x - 1 ? 1u : 0u;}
    __syncthreads();
    if (sc_last && tid == 0) {k3_publish_flags(P, st, dec, bufs.out);}
    return;
  }
  __syncthreads();

  // ---- phase 2: weighted column sums over this block's rows from shared memory, W[c] = sum_r w_r * (cs[c] + noise[r][c])
  const int stride = 3 * T + 2;
  float * part = bufs.partials + static_cast<size_t>(blockIdx.x) * stride;
  for (int c = tid; c < 3 * T; c += kUpdThreads) {
    const float cs_c = bufs.cs[c];
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    int r = 0;
    for (; r + 3 < rows_here; r += 4) {
      a0 = fmaf(s_w[r], __fadd_rn(cs_c, s_tile[static_cast<size_t>(r) * 3 * T + c]), a0);
      a1 = fmaf(s_w[r + 1], __fadd_rn(cs_c, s_tile[static_cast<size_t>(r + 1) * 3 * T + c]), a1);
      a2 = fmaf(s_w[r + 2], __fadd_rn(cs_c, s_tile[static_cast<size_t>(r + 2) * 3 * T + c]), a2);
      a3 = fmaf(s_w[r + 3], __fadd_rn(cs_c, s_tile[static_cast<size_t>(r + 3) * 3 * T + c]), a3);
    }
    for (; r < rows_here; ++r) {a0 = fmaf(s_w[r], __fadd_rn(cs_c, s_tile[static_cast<size_t>(r) * 3 * T + c]), a0);}
    part[2 + c] = (a0 + a1) + (a2 + a3);
  }
  if (tid == 0) {part[0] = s_stat[0]; part[1] = s_stat[1];}

  MPPI_TRACE_AT(20);
  // ---- phase 3: the last block to finish publishes the flags and, for small batches, merges all partials
  //      and writes the new control sequence (large batches: merge_finalize_kernel, launched by the host)
  __threadfence();
  __syncthreads();
  if (tid == 0) {sc_last = atomicAdd(&st->ticket, 1u) == gridDim.x - 1 ? 1u : 0u;}
  __syncthreads();
  if (!sc_last) {return;}
  __threadfence();
  MPPI_TRACE_AT(21);
  if (tid == 0) {k3_publish_flags(P, st, dec, bufs.out);}
  if (static_cast<int>(gridDim.x) > kLastBlockMergeMax) {return;}
  float * merged = bufs.rank_partial;   // [3T + 2]
  merge_partials(bufs.partials, gridDim.x, stride, T, inv_temp, merged, s_tile, tid, kUpdThreads);
  if (n_ranks <= 1) {
    __threadfence_block();
    __syncthreads();
    finalize_controls(P, merged, bufs.cs, bufs.out, tid, kUpdThreads);
  }
  MPPI_TRACE_AT(22);
}

// The tail of Optimizer::evalControl (optimizer.cpp:147-152) for one plane (0 vx, 1 vy, 2 wz) of the control sequence,
// v[T] in shared memory: utils::savitskyGolayFilter (utils.hpp:442-605) with the 4-deep control history (global, updated),
// getControlFromSequenceAsTwist (optimizer.cpp:396-410; returned) and shiftControlSequence (:206-225).  One thread; the
// filter is inherently sequential (already-filtered neighbours are reused) and reproduces the reference's quirks: index
// num_sequences - 4 is never filtered, vy is filtered for every model.
__device__ __forceinline__ float eval_tail_plane(float * v, float * __restrict__ hist, int plane, int T, int holonomic, int shift)
{
  const unsigned num_sequences = static_cast<unsigned>(T) - 1u;
  float h0 = hist[0 * 3 + plane], h1 = hist[1 * 3 + plane], h2 = hist[2 * 3 + plane], h3 = hist[3 * 3 + plane];
  if (num_sequences >= 20u) {
    float f[9] = {-21.0f, 14.0f, 39.0f, 54.0f, 59.0f, 54.0f, 39.0f, 14.0f, -21.0f};
#pragma unroll
    for (int i = 0; i < 9; ++i) {f[i] = __fdiv_rn(f[i], 231.0f);}
    auto apply = [&](float d0, float d1, float d2, float d3, float d4, float d5, float d6, float d7, float d8) -> float {
        float a = __fadd_rn(0.0f, __fmul_rn(d0, f[0]));
        a = __fadd_rn(a, __fmul_rn(d1, f[1])); a = __fadd_rn(a, __fmul_rn(d2, f[2])); a = __fadd_rn(a, __fmul_rn(d3, f[3]));
        a = __fadd_rn(a, __fmul_rn(d4, f[4])); a = __fadd_rn(a, __fmul_rn(d5, f[5])); a = __fadd_rn(a, __fmul_rn(d6, f[6]));
        a = __fadd_rn(a, __fmul_rn(d7, f[7])); a = __fadd_rn(a, __fmul_rn(d8, f[8]));
        return a;
      };
    unsigned idx = 0;
    v[idx] = apply(h0, h1, h2, h3, v[idx], v[idx + 1], v[idx + 2], v[idx + 3], v[idx + 4]);
    idx++;
    v[idx] = apply(h1, h2, h3, v[idx - 1], v[idx], v[idx + 1], v[idx + 2], v[idx + 3], v[idx + 4]);
    idx++;
    v[idx] = apply(h2, h3, v[idx - 2], v[idx - 1], v[idx], v[idx + 1], v[idx + 2], v[idx + 3], v[idx + 4]);
    idx++;
    v[idx] = apply(h3, v[idx - 3], v[idx - 2], v[idx - 1], v[idx], v[idx + 1], v[idx + 2], v[idx + 3], v[idx + 4]);
    for (idx = 4; idx != num_sequences - 4; idx++) {
      v[idx] = apply(v[idx - 4], v[idx - 3], v[idx - 2], v[idx - 1], v[idx], v[idx + 1], v[idx + 2], v[idx + 3], v[idx + 4]);
    }
    idx++;   // the reference's extra increment: index num_sequences - 4 stays unfiltered
    v[idx] = apply(v[idx - 4], v[idx - 3], v[idx - 2], v[idx - 1], v[idx], v[idx + 1], v[idx + 2], v[idx + 3], v[idx + 3]);
    idx++;
    v[idx] = apply(v[idx - 4], v[idx - 3], v[idx - 2], v[idx - 1], v[idx], v[idx + 1], v[idx + 2], v[idx + 2], v[idx + 2]);
    idx++;
    v[idx] = apply(v[idx - 4], v[idx - 3], v[idx - 2], v[idx - 1], v[idx], v[idx + 1], v[idx + 1], v[idx + 1], v[idx + 1]);
    idx++;
    v[idx] = apply(v[idx - 4], v[idx - 3], v[idx - 2], v[idx - 1], v[idx], v[idx], v[idx], v[idx], v[idx]);
    // control history: drop the oldest, append the command of this cycle
    const int offset = shift ? 1 : 0;
    hist[0 * 3 + plane] = h1; hist[1 * 3 + plane] = h2; hist[2 * 3 + plane] = h3; hist[3 * 3 + plane] = v[offset];
  }
  // getControlFromSequenceAsTwist: index 1 when the sequence is shifted afterwards, else 0; vy only if holonomic
  const float cmd = (plane == 1 && !holonomic) ? 0.0f : v[shift ? 1 : 0];
  if (shift && (plane != 1 || holonomic)) {
    // shiftControlSequence: roll by -1, then last = second to last (the old last element)
    const float last = v[T - 1];
    for (int t = 0; t + 1 < T; ++t) {v[t] = v[t + 1];}
    v[T - 1] = last;
  }
  return cmd;
}

// ---------------------------------------------------------------------------------------------------
// Fused small-batch kernel: K2, the furthest-point / survivor reduction, K3 and the merge in ONE cooperative launch.
// At the default 1000 x 56 the two-kernel cycle is bound by what surrounds the arithmetic: a launch boundary, a second
// cold start (record, path tables, noise rows requested again), K2's results making a round trip through global memory,
// and a serial per-trajectory walk of the path critics by one warp per block.  Here a block keeps its tile of 32
// trajectories in shared memory from the first noise load to the block's softmax record:
//   K2 body (rollout_tile_body, six planes: the noised controls survive beside x, y, yaw)
//   exchange 1         inside the GPU: one packet per tile (furthest-point candidate, survivor flags), collected by warp 0
//   decisions          (k3_decide, one thread)
//   path critics       one WARP per trajectory, lane = sampled pose (PathAlign, PathAlignLegacy) or time step (PathAngle);
//                      the two carried dependences of PathAlign (integrated distance, previous path point) run as
//                      shuffle chains of one add / one compare per sample, everything else is lane-parallel
//   totals, weights    warp 0, lane = trajectory, critic-list order with the fail_flag short-circuit + gamma term
//   weighted sums      all threads over the 3T columns, out of the tile
//   exchange 2         inside the GPU: the tile's softmax record leaves as packets
//   merge + clip       block t owns time steps t, t + G, ...: one warp per column over the records, redundant min;
//                      the result goes to device memory AND, as packets, straight into pinned host memory
// Both exchanges use the self-validating {value, tag} packets of the peer exchange (mppi_device.cuh): a packet whose tag
// equals the tag of this launch (*epoch + 1) is its own arrival flag, so there is no grid barrier, no fence and no atomic
// on the critical path.  The launch is cooperative: all blocks are co-resident, the bounded polls never time out in
// normal operation.
// ---------------------------------------------------------------------------------------------------
// PathAlignCritic::score (path_align_critic.cpp:92-135) for the 32 trajectories of the tile, by the whole block:
// lane = trajectory (every instruction serves 32 trajectories), and the sampled poses are dealt to the warps wherever the
// reference's loop carries nothing from one sample to the next.  The two carried dependences (the integrated distance
// and the previous path point) are walked by warp 0 alone: one add / one compare per sample.
//   A  all warps   segment length of every sampled pose (one IEEE sqrt each)
//   B  warp 0      traj_integrated_distance: the reference's sequential fp32 sum
//   -- independent of the furthest reached point up to here: runs while exchange 1 is in flight --
//   C  all warps   c = lower_bound(D[0, n), distance); utils::findClosestPathPt (utils.hpp:665-675) searches [init, n)
//                  with init = the previous answer: the answer is 0 when c <= init, else g = n - 1 (c == n) or the
//                  nearer of c - 1 and c.  c and g do not depend on init.
//   D  warp 0      the chain over init
//   E  all warps   distance to the chosen path point where it is valid
//   F  warp 0      mean over the valid samples, cost
__device__ __forceinline__ void path_align_distances(
  const DevParams * P, const FusedCtx & fx, int lane, int seg, int S)
{
  const int T = P->T, step = P->align_step;
  const int n_s = (T + step - 1) / step;     // sampled poses p = 0, step, 2 step, ... < T
  float * ad = fx.fs.ad;
  for (int k = 1 + seg; k < n_s; k += S) {
    const int o = k * step * kPad + lane;
    const float dxp = __fsub_rn(fx.s_x[o], fx.s_x[o - step * kPad]), dyp = __fsub_rn(fx.s_y[o], fx.s_y[o - step * kPad]);
    ad[k * kTile + lane] = __fsqrt_rn(__fadd_rn(__fmul_rn(dxp, dxp), __fmul_rn(dyp, dyp)));
  }
  __syncthreads();
  if (seg == 0) {
    float acc = 0.0f;
    for (int k0 = 1; k0 < n_s; k0 += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {v[u] = ad[min(k0 + u, n_s - 1) * kTile + lane];}
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k0 + u < n_s) {
          acc = __fadd_rn(acc, v[u]);
          ad[(k0 + u) * kTile + lane] = acc;
        }
      }
    }
  }
}

// phases C..F; the value returned to the lanes of warp 0 is the critic's term of trajectory `lane`.  Starts with a barrier
// of its own only where a phase needs the previous one (the caller has synchronised after the decisions).
__device__ __forceinline__ float path_align_finish(
  const DevParams * P, const FusedCtx & fx, int furthest, const float * path_yaw, int lane, int seg, int S)
{
  const int T = P->T, step = P->align_step;
  const int n_s = (T + step - 1) / step;
  const int n = furthest;                    // the arc-length prefix D[0, n) is searched
  const float * D = fx.fs.D;
  const float * ad = fx.fs.ad;
  int * ac = reinterpret_cast<int *>(fx.fs.ad + n_s * kTile);
  int top = 1;                               // largest power of two <= max(n, 1)
  while (top * 2 <= n) {top *= 2;}
  for (int k = 1 + seg; k < n_s; k += S) {
    const float mine = ad[k * kTile + lane];
    int c = 0;                               // number of prefix entries below the distance = lower_bound
    for (int bit = top; bit > 0; bit >>= 1) {
      const int probe = c + bit;
      if (probe <= n && D[probe - 1] < mine) {c = probe;}
    }
    int g = 0;
    if (c > 0) {
      if (c >= n) {
        g = n - 1;
      } else {
        g = __fsub_rn(mine, D[c - 1]) < __fsub_rn(D[c], mine) ? c - 1 : c;
      }
    }
    ac[k * kTile + lane] = c | (g << 16);    // both < 2^16
  }
  __syncthreads();
  if (seg == 0) {
    int prev = 0;
    for (int k0 = 1; k0 < n_s; k0 += 8) {
      int v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {v[u] = ac[min(k0 + u, n_s - 1) * kTile + lane];}
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k0 + u < n_s) {
          prev = (v[u] & 0xffff) <= prev ? 0 : (v[u] >> 16);
          ac[(k0 + u) * kTile + lane] = prev;
        }
      }
    }
  }
  __syncthreads();
  float psum = 0.0f, pnum = 0.0f;
  for (int k = 1 + seg; k < n_s; k += S) {
    const int res = ac[k * kTile + lane];
    if (fx.fs.valid[res]) {
      const int o = k * step * kPad + lane;
      const float dx = __fsub_rn(fx.fs.px[res], fx.s_x[o]), dy = __fsub_rn(fx.fs.py[res], fx.s_y[o]);
      pnum += 1.0f;
      // the distance itself only feeds the cost (1e-4 tolerance): one MUFU instead of the IEEE sequence
      if (P->align_use_yaw) {
        const float dyaw = static_cast<float>(normalize_angle_d(static_cast<double>(fx.s_yaw[o]) - static_cast<double>(path_yaw[res])));
        psum += sqrt_approx(dx * dx + dy * dy + dyaw * dyaw);
      } else {
        psum += sqrt_approx(dx * dx + dy * dy);
      }
    }
  }
  fx.fs.ap[(seg * 2) * kTile + lane] = psum;
  fx.fs.ap[(seg * 2 + 1) * kTile + lane] = pnum;
  __syncthreads();
  float term = 0.0f;
  if (seg == 0) {
    float summed = 0.0f, num = 0.0f;
    for (int w = 0; w < S; ++w) {summed += fx.fs.ap[(w * 2) * kTile + lane]; num += fx.fs.ap[(w * 2 + 1) * kTile + lane];}
    const float cost = num > 0.0f ? __fdiv_rn(summed, num) : 0.0f;
    term = add_pow_c(0.0f, __fmul_rn(cost, P->align.weight), P->align.power);
  }
  return term;
}

// The two per-warp path critics below are out of line, and they take the shared-memory planes and path tables by value:
// a FusedCtx passed by reference to a call would pin the whole record in local memory, and the tail would reload its
// pointers from there (an L1 round trip each, on the default path).
struct WarpCtx
{
  const float * s_x, * s_y, * s_yaw;   // time-major tile planes [T][33]
  const float * px, * py;              // path points
  const uint8_t * valid;
};
__device__ __forceinline__ WarpCtx warp_ctx(const FusedCtx & fx)
{
  return {fx.s_x, fx.s_y, fx.s_yaw, fx.fs.px, fx.fs.py, fx.fs.valid};
}

// PathAlignLegacyCritic::score (path_align_legacy_critic.cpp:97-128) for trajectory r, by one warp; lane = sampled pose
__device__ __noinline__ float path_align_legacy_warp(const DevParams * P, const WarpCtx fx, int r, const float * path_yaw, int lane)
{
  const int T = P->T, step = P->legacy_step, segs = P->N - 1;
  float summed = 0.0f;
  for (int p0 = step; p0 < T; p0 += 32 * step) {
    const int p = p0 + lane * step;
    float contrib = 0.0f;
    if (p < T) {
      const int o = p * kPad + r;
      const float Tx = fx.s_x[o], Ty = fx.s_y[o];
      const float Tyaw = P->legacy_use_yaw ? fx.s_yaw[o] : 0.0f;
      float min_d = 3.402823466e+38f;
      int min_s = 0;
      for (int sgm = 0; sgm < segs - 1; ++sgm) {
        const float dx = __fsub_rn(fx.px[sgm], Tx);
        const float dy = __fsub_rn(fx.py[sgm], Ty);
        float d = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        if (P->legacy_use_yaw) {
          const float dyaw = static_cast<float>(normalize_angle_d(static_cast<double>(Tyaw) - static_cast<double>(path_yaw[sgm])));
          d = __fadd_rn(d, __fmul_rn(dyaw, dyaw));
        }
        if (d < min_d) {min_d = d; min_s = sgm;}
      }
      if (min_s != 0 && fx.valid[min_s]) {contrib = __fsqrt_rn(min_d);}
    }
    summed += warp_sum(contrib);
  }
  const float evals = static_cast<float>(T / step);
  return add_pow_c(0.0f, __fmul_rn(__fdiv_rn(summed, evals), P->legacy.weight), P->legacy.power);
}

// PathAngleCritic::score (path_angle_critic.cpp:85-100) for trajectory r, by one warp; lane = time step
__device__ __noinline__ float path_angle_warp(const DevParams * P, const WarpCtx fx, int r, int angle_idx, int lane)
{
  const int T = P->T;
  const float gx = fx.px[angle_idx], gy = fx.py[angle_idx];
  float sum = 0.0f;
  for (int t = lane; t < T; t += 32) {
    const int o = t * kPad + r;
    const float x = fx.s_x[o], y = fx.s_y[o], yaw = fx.s_yaw[o];
    const float ybp = atan2f(__fsub_rn(gy, y), __fsub_rn(gx, x));
    double v = fabs(normalize_angle_d(static_cast<double>(__fsub_rn(ybp, yaw))));
    if (P->angle_reversing && !P->angle_forward_pref) {
      const double corrected = v < 1.57079632679489661923 ? static_cast<double>(ybp) :
        normalize_angle_d(static_cast<double>(ybp) + 3.14159265358979323846);
      v = fabs(normalize_angle_d(corrected - static_cast<double>(yaw)));
    }
    sum += static_cast<float>(v);
  }
  sum = warp_sum(sum);
  return add_pow_c(0.0f, (sum / static_cast<float>(T)) * P->angle.weight, P->angle.power);
}

__device__ __forceinline__ unsigned warp_or_u(unsigned v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {v |= __shfl_xor_sync(0xffffffffu, v, o);}
  return v;
}

// result packet for the host: pinned, mapped memory written straight from the kernel, {value, tag of the launch};
// the host polls the tags (finish_optimize), so no copy node, no stream synchronisation
__device__ __forceinline__ void put_result(float * out, uint2 * host_res, int idx, float v, unsigned tag)
{
  out[idx] = v;
  if (host_res) {st_packet(host_res + idx, __float_as_uint(v), tag);}
}

#ifndef MPPI_FUSED_MIN_BLOCKS
#define MPPI_FUSED_MIN_BLOCKS 2
#endif
// the work of one block on tile `tile` of `G` (blockIdx.x of gridDim.x; see the header comment above)
template<unsigned F, bool kExact>
__device__ __forceinline__ void tile_fused_body(
  const DevParams * Pg, const uint8_t * cm, const DevBuffers & bufs, const int B, const int T, const int n_cap,
  const int iteration, uint2 * host_res, const uint4 * up_host, const int up_vecs, const int tile, const int G,
  const int tail_mode, float * __restrict__ hist)
{
  // n_cap (path capacity, a multiple of 64) sizes the shared memory; the path size itself comes from the record, so a
  // captured graph survives the small changes of the pruned path from cycle to cycle
  __shared__ K3Decisions dec;
  __shared__ signed char s_src[kMaxCritics];
  FusedCtx fx;
  fx.n_cap = n_cap; fx.iteration = iteration;
  fx.up_host = up_host; fx.up_vecs = up_vecs;
  fx.tile = tile; fx.ntiles = G;
  const unsigned tag = ld_volatile_u32(bufs.epoch) + 1u;
  fx.tag = tag;
  rollout_tile_body<F, kExact, 0, true>(Pg, cm, bufs, B, T, &fx);

  const int S = blockDim.y, lane = threadIdx.x, seg = threadIdx.y;
  const int tid = seg * kTile + lane, nthr = S * kTile;
  const FusedShared & fs = fx.fs;
  const DevParams * P = reinterpret_cast<const DevParams *>(fx.s_hot);   // hot fields only
  DevState * st = bufs.st;
  const int b0 = tile * kTile;
  const int rows_here = min(kTile, B - b0);
  const int N = P->N;
  const float * path_yaw = reinterpret_cast<const float *>(Pg + 1) + 2 * N;   // written in this launch (zero-copy): coherent loads

  // PathAlign, the part that does not depend on the furthest reached point: done while exchange 1 is in flight
  if (P->align.on) {path_align_distances(P, fx, lane, seg, S);}

  // ---- exchange 1 inside the GPU: warp 0 collects every tile's packet (furthest-point candidate, survivor flags)
  if (seg == 0) {
    unsigned cand = 0u, flags = 0u;
    for (int i = lane; i < G; i += 32) {
      unsigned v;
      if (!poll_packet(bufs.pk_x1 + i, tag, v)) {raise_comm_error(bufs);}
      cand = max(cand, v & 0xffffu);
      flags |= v >> 16;
    }
    cand = warp_max_u(cand);
    flags = warp_or_u(flags);
    MPPI_TRACE_AT(10);
    // the decisions (k3_decide's logic on this launch's reductions), by every lane of warp 0 redundantly; lane q also
    // derives where the term of list position q comes from
    {
      const int nc = P->n_critics;
      int fail_at = nc;
      unsigned furthest = 0u;
      int fset = 0;
      if (iteration == 0) {
        fset = P->preset_furthest != kUnset; furthest = fset ? P->preset_furthest : 0u;
      } else {
        // carried over from the previous iteration's launch (critic_manager.cpp: fail_flag is only cleared in prepare())
        fset = st->furthest_set; furthest = st->furthest;
        if (st->fail_flag) {fail_at = -1;}
      }
      if (fail_at == nc) {
        // the first obstacle-type critic (list order) that saw no surviving trajectory raises fail_flag
        const int q0 = P->obstacle_q[0], q1 = P->obstacle_q[1];
        const bool ok0 = q0 == P->cost.idx ? (flags & 1u) != 0u : (flags & 2u) != 0u;
        const bool ok1 = q1 == P->cost.idx ? (flags & 1u) != 0u : (flags & 2u) != 0u;
        if (q0 >= 0 && !ok0) {
          fail_at = q0;
        } else if (q1 >= 0 && !ok1) {
          fail_at = q1;
        }
      }
      // the first enabled path critic in list order calls setPathFurthestPointIfNotSet (utils.hpp:350-355)
      if (!fset && P->first_path_q >= 0 && P->first_path_q <= fail_at) {furthest = cand; fset = 1;}
      const int f = min(static_cast<int>(furthest), N - 1);
      const unsigned gates = fs.flags[f];
      const int align_go = (P->align.on && P->align.idx <= fail_at && (gates & 1u)) ? 1 : 0;
      const int legacy_go = (P->legacy.on && P->legacy.idx <= fail_at && (gates & 2u)) ? 1 : 0;
      const int angle_go = (P->angle.on && P->angle.idx <= fail_at && (gates & 4u)) ? 1 : 0;
      if (lane == 0) {
        dec.fail_at = fail_at;
        dec.furthest = static_cast<int>(furthest);
        dec.furthest_set = fset;
        dec.follow_idx = (P->follow.on && P->follow.idx <= fail_at) ? fs.follow[f] : 0;
        dec.align_go = align_go; dec.legacy_go = legacy_go; dec.angle_go = angle_go;
        dec.angle_idx = min(static_cast<int>(furthest) + P->angle_offset, N - 1);
      }
      if (lane < nc) {
        int src = lane <= fail_at ? P->src_base[lane] : 0;
        if ((src == 3 && !align_go) || (src == 4 && !legacy_go) || (src == 5 && !angle_go)) {src = 0;}
        s_src[lane] = static_cast<signed char>(src);
      }
    }
  }
  __syncthreads();
  MPPI_TRACE_AT(11);

  // ---- path critics that need more than the end pose.  PathAlign: the whole block, lane = trajectory
  if (dec.align_go) {
    const float v = path_align_finish(P, fx, dec.furthest, path_yaw, lane, seg, S);
    if (seg == 0) {fs.term[1 * kTile + lane] = v;}
  }
  // PathAlignLegacy, PathAngle: one warp per trajectory
  if (dec.legacy_go || dec.angle_go) {
    for (int r = seg; r < rows_here; r += S) {
      if (dec.legacy_go) {
        const float v = path_align_legacy_warp(P, warp_ctx(fx), r, path_yaw, lane);
        if (lane == 0) {fs.term[2 * kTile + r] = v;}
      }
      if (dec.angle_go) {
        const float v = path_angle_warp(P, warp_ctx(fx), r, dec.angle_idx, lane);
        if (lane == 0) {fs.term[3 * kTile + r] = v;}
      }
    }
  }
  __syncthreads();
  MPPI_TRACE_AT(12);

  // ---- totals in critic-list order with the fail_flag short-circuit (critic_manager.cpp:67-76), gamma term,
  //      block-local softmax record (optimizer.cpp:362-391); warp 0, lane = trajectory.  s_src (made with the decisions)
  //      says where the term of list position q comes from: 0 nothing, 1 K2's row, 2.. the path critic terms.
  const float inv_temp = 1.0f / P->temperature;
  if (seg == 0) {
    const int b = b0 + lane;
    const bool live = b < B;
    const int nc = P->n_critics;
    float total = 3.402823466e+38f;
    if (live) {
      total = iteration == 0 ? 0.0f : bufs.costs[b];
      if (P->follow.on && P->follow.idx <= dec.fail_at) {    // path_follow_critic.cpp:60-70
        const float dx = fx.s_x[(T - 1) * kPad + lane] - fs.px[dec.follow_idx];
        const float dy = fx.s_y[(T - 1) * kPad + lane] - fs.py[dec.follow_idx];
        fs.term[lane] = add_pow_c(0.0f, P->follow.weight * sqrtf(dx * dx + dy * dy), P->follow.power);
      }
      for (int q = 0; q < nc; ++q) {
        const int src = s_src[q];
        if (src == 0) {continue;}
        const float term = src == 1 ? fs.rows[q * kTile + lane] : fs.term[(src - 2) * kTile + lane];
        total = __fadd_rn(total, term);
      }
      if (P->want_critic_rows) {
        // per-critic getter (mppi_get_critic_costs): path critic rows come from here, rows of critics that did not
        // run read as zero
        float * rows = bufs.crit_rows;
        for (int q = 0; q < nc; ++q) {
          const int src = s_src[q];
          if (src >= 2) {
            rows[static_cast<size_t>(q) * B + b] = fs.term[(src - 2) * kTile + lane];
          } else if (src == 0) {
            rows[static_cast<size_t>(q) * B + b] = 0.0f;
          }
        }
      }
      // gamma term (optimizer.cpp:367-380): vx, then wz, then vy (holonomic)
      total = __fadd_rn(total, __fmul_rn(P->gamma_vx, fs.rows[nc * kTile + lane]));
      total = __fadd_rn(total, __fmul_rn(P->gamma_wz, fs.rows[(nc + 2) * kTile + lane]));
      if (P->holonomic) {total = __fadd_rn(total, __fmul_rn(P->gamma_vy, fs.rows[(nc + 1) * kTile + lane]));}
      bufs.costs[b] = total;
    }
    // optimizer.cpp:382-391 on this tile: m = min, w = exp(-(c - m) / temperature), s = sum w
    const float m = warp_min(total);
    const float w_b = live ? expf(-(total - m) * inv_temp) : 0.0f;
    const float ssum = warp_sum(w_b);
    fs.w[lane] = w_b;
    if (lane == 0) {fs.stat[0] = m; fs.stat[1] = ssum;}
  }
  __syncthreads();
  MPPI_TRACE_AT(13);

  // ---- weighted column sums of the tile, W[c] = sum_r w_r * c[r][c], out of the noised controls still in the tile;
  //      the record leaves as packets (exchange 2 inside the GPU)
  const int stride = 3 * T + 2;
  uint2 * part = bufs.pk_rec + static_cast<size_t>(tile) * stride;
  if (tid == 0) {st_packet(part, __float_as_uint(fs.stat[0]), tag);}
  if (tid == 32 || (S == 1 && tid == 1)) {st_packet(part + 1, __float_as_uint(fs.stat[1]), tag);}
  for (int c = tid; c < 3 * T; c += nthr) {
    const int plane = c / T, t = c - plane * T;
    const float * col = (plane == 0 ? fx.s_cvx : (plane == 1 ? fx.s_cvy : fx.s_cwz)) + t * kPad;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    int r = 0;
    for (; r + 3 < rows_here; r += 4) {
      a0 = fmaf(fs.w[r], col[r], a0);
      a1 = fmaf(fs.w[r + 1], col[r + 1], a1);
      a2 = fmaf(fs.w[r + 2], col[r + 2], a2);
      a3 = fmaf(fs.w[r + 3], col[r + 3], a3);
    }
    for (; r < rows_here; ++r) {a0 = fmaf(fs.w[r], col[r], a0);}
    st_packet(part + 2 + c, __float_as_uint((a0 + a1) + (a2 + a3)), tag);
  }
  MPPI_TRACE_AT(14);

  // ---- merge + clip: block t owns time steps t, t + G, ...  It needs m and s of every record and its own columns;
  //      the polls return as soon as the packets of this launch are there (no barrier)
  // tail_mode != 0 (mppi_eval_control): the owners hand their time steps to tile 0 as packets instead of writing them out;
  // tile 0 runs the evalControl tail on the whole sequence and delivers the result (below)
  const bool tail = tail_mode != 0;
  if (tile == 0 && tid == 0) {
    k3_publish_flags(P, st, dec, bufs.out);
    if (host_res) {
      st_packet(host_res + 3 * T, static_cast<unsigned>(st->fail_flag), tag);
      st_packet(host_res + 3 * T + 1, dec.furthest_set ? static_cast<unsigned>(dec.furthest) : kUnset, tag);
    }
    *bufs.epoch = tag;     // every block read the epoch before block 0 can get here (it needs a packet of every block)
  }
  if (tile >= T) {return;}   // owns no time step
  const uint2 * recs = bufs.pk_rec;
  const bool small = G <= 32;   // one record per lane: every warp rescales on its own, one memory round trip in all
  float m = 3.402823466e+38f;
  if (!small) {
    for (int i = tid; i < G; i += nthr) {
      unsigned bits;
      if (!poll_packet(recs + static_cast<size_t>(i) * stride, tag, bits)) {raise_comm_error(bufs);}
      const float mi = __uint_as_float(bits);
      fs.e[i] = mi;
      m = fminf(m, mi);
    }
    m = warp_min(m);
    if (lane == 0) {fs.red[seg] = m;}
    __syncthreads();
    m = fs.red[0];
    for (int w = 1; w < S; ++w) {m = fminf(m, fs.red[w]);}
    __syncthreads();
    for (int i = tid; i < G; i += nthr) {fs.e[i] = expf(-(fs.e[i] - m) * inv_temp);}
    __syncthreads();
  }
  // column 0 = sum of the weights; then (vx, vy, wz) of every owned time step: one warp per column, lanes over the records
  const int n_own = (T - tile + G - 1) / G;
  float * col_out = fs.red + 8;   // [1 + 3 * 7]
  for (int t_base = 0; t_base < n_own; t_base += 7) {
    const int n_now = min(7, n_own - t_base);
    for (int k = seg; k < 1 + 3 * n_now; k += S) {
      int col;
      if (k == 0) {
        col = 0;
      } else {
        const int t = tile + (t_base + (k - 1) / 3) * G, plane = (k - 1) % 3;
        col = 1 + plane * T + t;
      }
      float acc = 0.0f;
      if (small) {
        // lane = record: its minimum and its entry of this column are polled together
        float mi = 3.402823466e+38f, wi = 0.0f;
        if (lane < G) {
          const uint2 * pm = recs + static_cast<size_t>(lane) * stride;
          const long long t0 = clock64();
          for (;;) {
            const uint2 a = ld_packet(pm), w = ld_packet(pm + 1 + col);
            if (a.y == tag && w.y == tag) {mi = __uint_as_float(a.x); wi = __uint_as_float(w.x); break;}
            if (clock64() - t0 > kSpinLimitCycles) {raise_comm_error(bufs); mi = 0.0f; break;}
          }
        }
        const float mm = warp_min(mi);
        acc = lane < G ? wi * expf(-(mi - mm) * inv_temp) : 0.0f;
      } else {
        for (int i = lane; i < G; i += 32) {
          unsigned bits;
          if (!poll_packet(recs + static_cast<size_t>(i) * stride + 1 + col, tag, bits)) {raise_comm_error(bufs);}
          acc = fmaf(__uint_as_float(bits), fs.e[i], acc);
        }
      }
      acc = warp_sum(acc);
      if (lane == 0) {col_out[k] = acc;}
    }
    __syncthreads();
    if (tid < n_now) {
      // cs = W / sum, then applyControlSequenceConstraints (optimizer.cpp:237-249)
      const int t = tile + (t_base + tid) * G;
      const float ssum = col_out[0];
      float vx = col_out[1 + 3 * tid] / ssum, wz = col_out[3 + 3 * tid] / ssum, vy = fx.s_cs[T + t];
      if (P->holonomic) {
        vy = col_out[2 + 3 * tid] / ssum;
        vy = fminf(fmaxf(vy, -P->c_vy), P->c_vy);
      }
      vx = fminf(fmaxf(vx, P->c_vx_min), P->c_vx_max);
      wz = fminf(fmaxf(wz, -P->c_wz), P->c_wz);
      if (P->model == MPPI_MODEL_ACKERMANN) {   // motion_models.hpp:110-117
        const float rr = P->min_turning_r;
        if (fabsf(vx) / fabsf(wz) < rr) {
          const float sgn = wz > 0.0f ? 1.0f : (wz < 0.0f ? -1.0f : 0.0f);
          wz = sgn * fabsf(vx) / rr;
        }
      }
      if (tail) {
        st_packet(bufs.pk_out + t, __float_as_uint(vx), tag);
        st_packet(bufs.pk_out + T + t, __float_as_uint(vy), tag);
        st_packet(bufs.pk_out + 2 * T + t, __float_as_uint(wz), tag);
      } else {
        bufs.cs[t] = vx; bufs.cs[T + t] = vy; bufs.cs[2 * T + t] = wz;
        put_result(bufs.out, host_res, t, vx, tag);
        put_result(bufs.out, host_res, T + t, vy, tag);
        put_result(bufs.out, host_res, 2 * T + t, wz, tag);
      }
    }
    __syncthreads();
  }
  MPPI_TRACE_AT(15);
  if (tail && tile == 0) {
    // ---- the tail of evalControl (Savitzky-Golay filter, command, shift) on the whole new sequence: exchange 3 inside the
    //      GPU collects it from the owners; skipped when the optimisation failed (the reference only reaches this code
    //      after fallback() returned false)
    float * v = const_cast<float *>(fx.s_cvx);   // the tile planes are free now: [3][T]
    for (int i = tid; i < 3 * T; i += nthr) {
      unsigned bits;
      if (!poll_packet(bufs.pk_out + i, tag, bits)) {raise_comm_error(bufs);}
      v[i] = __uint_as_float(bits);
    }
    __syncthreads();
    const bool failed = dec.fail_at < P->n_critics;
    if (tid < 3) {
      float cmd = 0.0f;
      if (!failed) {cmd = eval_tail_plane(v + tid * T, hist, tid, T, P->holonomic, tail_mode == 2 ? 1 : 0);}
      put_result(bufs.out, host_res, 3 * T + 2 + tid, cmd, tag);
    }
    __syncthreads();
    for (int i = tid; i < 3 * T; i += nthr) {
      bufs.cs[i] = v[i];
      put_result(bufs.out, host_res, i, v[i], tag);
    }
  }
}

// (Pg, cm: no __restrict__ -- the tiles write both during the zero-copy upload)
// kDevMap: see rollout_score_kernel (never with the zero-copy upload: the record is in device memory before the launch)
template<unsigned F, bool kExact, bool kDevMap = false>
__global__ void __launch_bounds__(256, MPPI_FUSED_MIN_BLOCKS) tile_fused_kernel(
  const DevParams * Pg, const uint8_t * cm, DevBuffers bufs, const int B, const int T, const int n_cap,
  const int iteration, uint2 * host_res, const uint4 * up_host, const int up_vecs, const int tail_mode, float * hist)
{
  tile_fused_body<F, kExact>(Pg, kDevMap ? Pg->cm_dev : cm, bufs, B, T, n_cap, iteration, host_res, up_host, up_vecs, blockIdx.x,
    gridDim.x, tail_mode, hist);
}

// K3c (stream layout): softmax weights and weighted control sums over time-major noise [T][B]; a GEMV
// W[c] = sum_b w_b * (cs[c] + noise[c][b]) that is pure HBM streaming (12 B per rollout step).
// One block owns kWsChunk consecutive trajectories.  Every warp keeps the weights of the WHOLE chunk in
// registers (lane owns kWsVec groups of 4 consecutive b: 16-byte loads, coalesced along b) and walks the
// (plane, t) rows warp, warp + 8, ...: kWsVec independent 16-byte loads in flight per lane, one shuffle
// reduction per row, no shared memory, no barriers.  The rows are split over gridDim.y so that small chunk
// counts still fill the machine.  The record written per chunk is [m = global min, s, W...] so that
// merge_finalize_kernel merges it like any other partial.
constexpr int kWsThreads = 256;
constexpr int kWsVec = 8;
constexpr int kWsChunk = 32 * 4 * kWsVec;   // 1024 trajectories per block

__device__ __forceinline__ void weighted_sums_tm_body(const DevParams * __restrict__ Pg, const DevBuffers & bufs)
{
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_launch_dependents();
  pdl_wait();
  const int T = Pg->T, B = Pg->B;
  const float inv_temp = 1.0f / Pg->temperature;
  const float gm = bufs.st->global_min;
  const int stride = 3 * T + 2;
  float * part = bufs.partials + static_cast<size_t>(blockIdx.x) * stride;
  const int b0 = blockIdx.x * kWsChunk + lane * 4;
  const bool full = (B & 3) == 0 && blockIdx.x * kWsChunk + kWsChunk <= B;   // whole chunk in range, rows 16-byte aligned
  float w[kWsVec][4];
  float ssum = 0.0f;
#pragma unroll
  for (int i = 0; i < kWsVec; ++i) {
    const int b = b0 + i * 128;
    float c[4];
    if (full) {
      const float4 v = __ldg(reinterpret_cast<const float4 *>(bufs.costs + b));
      c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {c[j] = b + j < B ? __ldg(bufs.costs + b + j) : 0.0f;}
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      w[i][j] = (full || b + j < B) ? expf(-(c[j] - gm) * inv_temp) : 0.0f;
      ssum += w[i][j];
    }
  }
  if (blockIdx.y == 0 && warp == 0) {
    ssum = warp_sum(ssum);
    if (lane == 0) {part[0] = gm; part[1] = ssum;}
  }
  const int rows_total = 3 * T;
  const int rows_per = (rows_total + static_cast<int>(gridDim.y) - 1) / static_cast<int>(gridDim.y);
  const int c_begin = blockIdx.y * rows_per, c_end = min(rows_total, c_begin + rows_per);
  for (int c = c_begin + warp; c < c_end; c += kWsThreads / 32) {
    const int plane = c / T, t = c - plane * T;
    const float * __restrict__ row = (plane == 0 ? bufs.in_a : (plane == 1 ? bufs.in_b : bufs.in_c)) + static_cast<size_t>(t) * B + b0;
    const float cs_t = bufs.cs[c];
    float acc0 = 0.0f, acc1 = 0.0f;
    if (full) {
      float4 v[kWsVec];
#pragma unroll
      for (int i = 0; i < kWsVec; ++i) {v[i] = __ldg(reinterpret_cast<const float4 *>(row + i * 128));}
#pragma unroll
      for (int i = 0; i < kWsVec; i += 2) {
        acc0 = fmaf(w[i][0], __fadd_rn(cs_t, v[i].x), acc0);
        acc0 = fmaf(w[i][1], __fadd_rn(cs_t, v[i].y), acc0);
        acc0 = fmaf(w[i][2], __fadd_rn(cs_t, v[i].z), acc0);
        acc0 = fmaf(w[i][3], __fadd_rn(cs_t, v[i].w), acc0);
        acc1 = fmaf(w[i + 1][0], __fadd_rn(cs_t, v[i + 1].x), acc1);
        acc1 = fmaf(w[i + 1][1], __fadd_rn(cs_t, v[i + 1].y), acc1);
        acc1 = fmaf(w[i + 1][2], __fadd_rn(cs_t, v[i + 1].z), acc1);
        acc1 = fmaf(w[i + 1][3], __fadd_rn(cs_t, v[i + 1].w), acc1);
      }
    } else {
#pragma unroll
      for (int i = 0; i < kWsVec; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (b0 + i * 128 + j < B) {acc0 = fmaf(w[i][j], __fadd_rn(cs_t, __ldg(row + i * 128 + j)), acc0);}
        }
      }
    }
    const float a = warp_sum(acc0 + acc1);
    if (lane == 0) {part[2 + c] = a;}
  }
}

__global__ void __launch_bounds__(kWsThreads) weighted_sums_tm_kernel(const DevParams * __restrict__ Pg, DevBuffers bufs)
{
  weighted_sums_tm_body(Pg, bufs);
}

// ---------------------------------------------------------------------------------------------------
// K3c, Blackwell data path (stream layout, B % 4 == 0): the weighted control sums W[c] = sum_b w_b (cs[c] + noise[c][b])
// with the noise streamed through shared memory by the TMA unit instead of per-lane 16-byte loads (optimizer.cpp:384-391).
//
// One block owns kPsChunk = 1024 consecutive trajectories (columns of the time-major planes) and a range of row groups
// (gridDim.y).  The last warp is the PRODUCER: its first lane fills a ring of kPsStages stages with cp.async.bulk.tensor.2d
// (a stage = 4 rows x 1024 columns = 16 KB as four boxes of 4 x 256, completion counted on the stage's `full` mbarrier)
// before anything else happens in the block, and refills a stage as soon as the 4 consumer warps have released it (`empty`
// mbarrier).  The CONSUMERS turn the block's 1024 costs into weights (32 per lane, in registers) while the first stages are in
// flight, then drain the ring: warp w owns row w of every stage, eight conflict-free 16-byte shared loads per lane, 32 FMAs,
// one shuffle reduction per row.  No __syncthreads in the steady state; 64 KB in flight per block whatever the consumers
// do, which is what the register-staged version lacked (long-scoreboard 25 per issue at 41 % occupancy, profiles/r01b).  Columns beyond B
// are zero-filled by the TMA unit (their weights are zero too).  Chunks are taken in DESCENDING column order (the columns the
// rollout kernel read last); at 262144 x 100 DRAM still delivers all 317 MB - the path-cost kernel's 65 MB in between
// evict them - so the order is harmless, not a gain.  Every block pays the same start-up before its first row (1024 costs ->
// 32 exponentials per lane, all eight loads of a lane in flight at once), so the host picks FEW row groups (about 2.5 blocks
// per SM in all).  The record per chunk is [m = global min, s, W[3T]]; on one rank the block that finishes a row group last
// merges that group's columns itself (below), otherwise merge_finalize_kernel / merge_exchange_finalize_kernel follow.
// ---------------------------------------------------------------------------------------------------
constexpr int kPsChunk = 1024;            // trajectories (columns) per block
constexpr int kPsBoxCols = 256;           // columns per TMA box (the hardware limit of a box dimension)
constexpr int kPsSub = kPsChunk / kPsBoxCols;
constexpr int kPsRows = 4;                // rows per stage == consumer warps
#ifndef MPPI_PS_STAGES
#define MPPI_PS_STAGES 4
#endif
constexpr int kPsStages = MPPI_PS_STAGES;
constexpr int kPsConsumers = 32 * kPsRows;
constexpr int kPsThreads = kPsConsumers + 32;
constexpr int kPsBoxBytes = kPsRows * kPsBoxCols * 4;
constexpr int kPsStageBytes = kPsSub * kPsBoxBytes;
constexpr int kWsDoneSlots = 1024;       // row-group counters of the fused merge; the last one counts finished row groups
constexpr int kPsSpinLimit = 1 << 22;     // bounded mbarrier waits (each try_wait suspends the thread for a while)

__host__ __device__ inline size_t ps_smem_bytes() {return static_cast<size_t>(kPsStages) * kPsStageBytes + 128;}

__device__ __forceinline__ unsigned smem_u32(const void * p) {return static_cast<unsigned>(__cvta_generic_to_shared(p));}
__device__ __forceinline__ void mbar_init(uint64_t * bar, unsigned count)
{
  asm volatile ("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t * bar)
{
  asm volatile ("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t * bar, unsigned bytes)
{
  asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded wait for the phase with the given parity; false on time-out
__device__ __forceinline__ bool mbar_wait(uint64_t * bar, unsigned parity)
{
  const unsigned a = smem_u32(bar);
#pragma unroll 1
  for (int spin = 0; spin < kPsSpinLimit; ++spin) {
    unsigned done;
    asm volatile (
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(a), "r"(parity) : "memory");
    if (done) {return true;}
  }
  return false;
}
__device__ __forceinline__ void tma_load_2d(void * dst, const CUtensorMap * map, int col, int row, uint64_t * bar)
{
  asm volatile (
    "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
    :: "r"(smem_u32(dst)), "l"(reinterpret_cast<unsigned long long>(map)), "r"(col), "r"(row), "r"(smem_u32(bar)) : "memory");
}

// one stage = kPsRows rows x kPsChunk columns as kPsSub boxes side by side (box q lands at q * kPsBoxBytes): the four boxes of
// a stage ask for the same rows back to back, so DRAM sees 4 KB contiguous per row like the register-staged kernel
__device__ __forceinline__ void ps_fill_stage(float * stage, const CUtensorMap * map, int b0, int t0, uint64_t * bar)
{
  mbar_arrive_expect_tx(bar, kPsStageBytes);
#pragma unroll
  for (int q = 0; q < kPsSub; ++q) {tma_load_2d(stage + q * (kPsBoxBytes / 4), map, b0 + q * kPsBoxCols, t0, bar);}
}

__global__ void __launch_bounds__(kPsThreads) weighted_sums_tma_kernel(
  const __grid_constant__ CUtensorMap tm_vx, const __grid_constant__ CUtensorMap tm_vy, const __grid_constant__ CUtensorMap tm_wz,
  const DevParams * __restrict__ Pg, DevBuffers bufs, const int T, const int B, const int holonomic,
  unsigned * __restrict__ done, uint2 * host_res)
{
  extern __shared__ __align__(128) float ps_smem[];
  __shared__ __align__(8) uint64_t s_full[kPsStages], s_empty[kPsStages];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float * s_stage = ps_smem;
  // grid = (chunks, row groups); chunks in DESCENDING order (see above)
  const int n_chunks = static_cast<int>(gridDim.x), n_groups = static_cast<int>(gridDim.y);
  const int group = static_cast<int>(blockIdx.y);
  const int chunk = n_chunks - 1 - static_cast<int>(blockIdx.x);
  const int b0 = chunk * kPsChunk;
  // stages in ring order: plane vx, plane wz, [plane vy]; this block's share of them (gridDim.y row groups)
  const int boxes_per_plane = (T + kPsRows - 1) / kPsRows;
  const int n_all = (holonomic ? 3 : 2) * boxes_per_plane;
  const int per_y = (n_all + n_groups - 1) / n_groups;
  const int box_begin = group * per_y, n_boxes = max(0, min(n_all, box_begin + per_y) - box_begin);
  pdl_launch_dependents();

  if (tid == kPsConsumers) {
    for (int s = 0; s < kPsStages; ++s) {mbar_init(&s_full[s], 1u); mbar_init(&s_empty[s], kPsConsumers / 32);}
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
    for (int i = 0; i < min(kPsStages, n_boxes); ++i) {
      const int g = box_begin + i, pl = g / boxes_per_plane, t0 = (g - pl * boxes_per_plane) * kPsRows;
      ps_fill_stage(s_stage + i * (kPsStageBytes / 4), pl == 0 ? &tm_vx : (pl == 1 ? &tm_wz : &tm_vy), b0, t0, &s_full[i]);
    }
  }
  __syncthreads();     // the barriers are initialised for everybody

  if (warp == kPsConsumers / 32) {
    if (lane == 0) {
      for (int i = kPsStages; i < n_boxes; ++i) {
        const int s = i % kPsStages;
        if (!mbar_wait(&s_empty[s], ((i / kPsStages) - 1) & 1u)) {raise_comm_error(bufs); break;}   // the stage's previous use is drained
        const int g = box_begin + i, pl = g / boxes_per_plane, t0 = (g - pl * boxes_per_plane) * kPsRows;
        ps_fill_stage(s_stage + s * (kPsStageBytes / 4), pl == 0 ? &tm_vx : (pl == 1 ? &tm_wz : &tm_vy), b0, t0, &s_full[s]);
      }
    }
    return;
  }
  // ---- consumers: softmax weights of the chunk; lane owns columns q * 256 + j * 128 + 4 lane + {0..3}, q < 4, j < 2
  //      (the noise planes are static, the costs and their minimum are the path-cost kernel's: wait for it here, with the
  //       first stages of the ring already in flight)
  const float inv_temp = 1.0f / Pg->temperature;
  pdl_wait();
  const float gm = __ldcg(&bufs.st->global_min);
  float w[kPsSub][2][4];
  float ssum = 0.0f;
#pragma unroll
  for (int q = 0; q < kPsSub; ++q) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int b = b0 + q * kPsBoxCols + j * 128 + 4 * lane;
      float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      if (b + 3 < B) {
        const float4 v = __ldcg(reinterpret_cast<const float4 *>(bufs.costs + b));   // the lane's eight loads are all in flight before the first exponential
        c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {if (b + e < B) {c[e] = __ldcg(bufs.costs + b + e);}}
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {w[q][j][e] = c[e];}
    }
  }
#pragma unroll
  for (int q = 0; q < kPsSub; ++q) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        w[q][j][e] = b0 + q * kPsBoxCols + j * 128 + 4 * lane + e < B ? expf(-(w[q][j][e] - gm) * inv_temp) : 0.0f;
        ssum += w[q][j][e];
      }
    }
  }
  ssum = warp_sum(ssum);          // every warp holds the whole chunk: the same sum in every warp
  float * part = bufs.partials + static_cast<size_t>(chunk) * (3 * T + 2);
  // every row group writes the head of the record (the same bits from every group: each holds the whole chunk's weights), so
  // that the group that merges its own columns (below) depends on the blocks of its own group only
  if ((group == 0 || done != nullptr) && tid == 0) {part[0] = gm; part[1] = ssum;}
  for (int i = 0; i < n_boxes; ++i) {
    const int s = i % kPsStages;
    if (!mbar_wait(&s_full[s], (i / kPsStages) & 1u)) {raise_comm_error(bufs); break;}
    const int g = box_begin + i, pl = g / boxes_per_plane, t = (g - pl * boxes_per_plane) * kPsRows + warp;
    const float * row = s_stage + s * (kPsStageBytes / 4) + warp * kPsBoxCols + 4 * lane;
    float4 v[kPsSub][2];
#pragma unroll
    for (int q = 0; q < kPsSub; ++q) {
      v[q][0] = *reinterpret_cast<const float4 *>(row + q * (kPsBoxBytes / 4));
      v[q][1] = *reinterpret_cast<const float4 *>(row + q * (kPsBoxBytes / 4) + 128);
    }
    __syncwarp();
    if (lane == 0) {mbar_arrive(&s_empty[s]);}
    float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
    for (int q = 0; q < kPsSub; ++q) {
      a0 = fmaf(w[q][0][0], v[q][0].x, a0); a1 = fmaf(w[q][1][0], v[q][1].x, a1);
      a0 = fmaf(w[q][0][1], v[q][0].y, a0); a1 = fmaf(w[q][1][1], v[q][1].y, a1);
      a0 = fmaf(w[q][0][2], v[q][0].z, a0); a1 = fmaf(w[q][1][2], v[q][1].z, a1);
      a0 = fmaf(w[q][0][3], v[q][0].w, a0); a1 = fmaf(w[q][1][3], v[q][1].w, a1);
    }
    const float a = warp_sum(a0 + a1);
    if (lane == 0 && t < T) {
      const int c = (pl == 0 ? 0 : (pl == 1 ? 2 : 1)) * T + t;       // record order: vx, vy, wz
      part[2 + c] = fmaf(__ldcg(bufs.cs + c), ssum, a);              // sum_b w_b (cs + noise) = cs * s + sum_b w_b noise
    }
  }
  if (done == nullptr) {return;}
  // ---- merge + normalise + clip (optimizer.cpp:384-394, :237-249) without another kernel: the block that finishes a row
  //      group LAST sums that group's columns over all chunks (every record carries the same minimum - the global one - so
  //      the online-softmax merge is a plain sum, taken in the order merge_finalize_kernel takes it), divides by the
  //      normaliser, clips and delivers its part of the new control sequence (device memory and, when asked, result packets
  //      in pinned host memory).  Row groups finish at different times: their merges hide behind the other groups' streaming.
  __shared__ unsigned s_last;
  __threadfence();
  asm volatile ("bar.sync 1, %0;" :: "n"(kPsConsumers) : "memory");
  if (tid == 0) {s_last = atomicAdd(&done[group], 1u) == static_cast<unsigned>(n_chunks) - 1u ? 1u : 0u;}
  asm volatile ("bar.sync 1, %0;" :: "n"(kPsConsumers) : "memory");
  if (!s_last) {return;}
  __threadfence();
  const int stride = 3 * T + 2;
  const float * parts = bufs.partials;
  const unsigned tag = host_res ? ld_volatile_u32(bufs.epoch) : 0u;
  // thread = column of the row group, all chunks in chunk order (four interleaved partial sums: a fixed order); the loads
  // of a thread are independent, consecutive threads read consecutive words
  for (int r = tid; r < n_boxes * kPsRows; r += kPsConsumers) {
    const int g = box_begin + r / kPsRows, pl = g / boxes_per_plane, t = (g - pl * boxes_per_plane) * kPsRows + r % kPsRows;
    if (t >= T) {continue;}
    const int plane = pl == 0 ? 0 : (pl == 1 ? 2 : 1), c = plane * T + t;
    float a[4] = {0.0f, 0.0f, 0.0f, 0.0f}, sw[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    const float * p0 = parts + 2 + c;
    int i = 0;
    for (; i + 16 <= n_chunks; i += 16) {   // 32 loads of the thread in flight: the merge is a few L2 round trips
      float va[16], vs[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        va[u] = __ldcg(p0 + static_cast<size_t>(i + u) * stride);
        vs[u] = __ldcg(parts + static_cast<size_t>(i + u) * stride + 1);
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {a[u & 3] += va[u]; sw[u & 3] += vs[u];}
    }
    for (; i + 4 <= n_chunks; i += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        a[u] += __ldcg(p0 + static_cast<size_t>(i + u) * stride);
        sw[u] += __ldcg(parts + static_cast<size_t>(i + u) * stride + 1);
      }
    }
    for (; i < n_chunks; ++i) {a[0] += __ldcg(p0 + static_cast<size_t>(i) * stride); sw[0] += __ldcg(parts + static_cast<size_t>(i) * stride + 1);}
    const float acc = (a[0] + a[1]) + (a[2] + a[3]), S = (sw[0] + sw[1]) + (sw[2] + sw[3]);
    float v = acc / S;
    if (plane == 0) {
      v = fminf(fmaxf(v, Pg->c_vx_min), Pg->c_vx_max);
    } else if (plane == 1) {
      v = fminf(fmaxf(v, -Pg->c_vy), Pg->c_vy);
    } else {
      v = fminf(fmaxf(v, -Pg->c_wz), Pg->c_wz);
    }
    bufs.cs[c] = v; bufs.out[c] = v;
    if (host_res) {st_packet(host_res + c, __float_as_uint(v), tag);}
  }
  if (group == 0) {
    // what no row group owns: the lateral plane of a non-holonomic model (unchanged), the fail flag and the furthest
    // reached path point (published by the path-cost kernel in front of this one)
    if (!holonomic) {
      for (int t = tid; t < T; t += kPsConsumers) {
        const float vy = bufs.cs[T + t];
        bufs.out[T + t] = vy;
        if (host_res) {st_packet(host_res + T + t, __float_as_uint(vy), tag);}
      }
    }
    if (host_res && tid == 0) {
      st_packet(host_res + 3 * T, __float_as_uint(bufs.out[3 * T]), tag);
      st_packet(host_res + 3 * T + 1, __float_as_uint(bufs.out[3 * T + 1]), tag);
    }
  }
  if (tid == 0) {done[group] = 0u;}   // ready for the next launch (nobody else touches this group's counter any more)
}

// K4: parallel merge of n partial records [m, s, W...] (online-softmax merge, SURVEY 8e exchange 2).
// Used (a) after K3 when the batch produced more partials than one block should merge serially, and
// (b) in sharded configurations on the all-gathered per-rank records; every rank merges redundantly and
// applies the clip, so no broadcast is needed afterwards.  One block owns kMergeT time steps (3 columns each)
// and all its threads stride over the partials; `finalize` = 0 writes the merged record to dst instead.

constexpr int kMergeCached = 2048;   // partial records whose rescale factors are cached in shared memory

// host_res != nullptr (finalize only): the result also goes straight into pinned host memory as {value, tag} packets
// (multi-robot groups: no copy node and no stream synchronisation per robot, see wait_result_packets)
__device__ __forceinline__ void merge_finalize_body(
  const DevParams * __restrict__ Pg, const float * __restrict__ parts, int n, int stride, const DevBuffers & bufs, int finalize,
  float * __restrict__ dst, uint2 * host_res, unsigned tag)
{
  __shared__ float s_red[kUpdThreads / 32];
  __shared__ float s_col[3 * kMergeT + 1];
  __shared__ float s_e[kMergeCached];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = Pg->T;
  const float inv_temp = 1.0f / Pg->temperature;
  // global minimum over the partials
  float m = 3.402823466e+38f;
  for (int i = tid; i < n; i += kUpdThreads) {m = fminf(m, __ldg(parts + static_cast<size_t>(i) * stride));}
  m = warp_min(m);
  if (lane == 0) {s_red[warp] = m;}
  __syncthreads();
  m = s_red[0];
#pragma unroll
  for (int w = 1; w < kUpdThreads / 32; ++w) {m = fminf(m, s_red[w]);}
  // rescale factor of every record, once
  for (int i = tid; i < min(n, kMergeCached); i += kUpdThreads) {
    s_e[i] = expf(-(__ldg(parts + static_cast<size_t>(i) * stride) - m) * inv_temp);
  }
  __syncthreads();
  const int t_first = blockIdx.x * kMergeT;
  // column 0 = sum of weights, then (vx, vy, wz) of each owned time step; one warp per column, lanes over the records
  for (int k = warp; k < 3 * kMergeT + 1; k += kUpdThreads / 32) {
    int col;   // index into the record after the leading m: 0 = s, 1 + plane * T + t = W
    if (k == 0) {
      col = 0;
    } else {
      const int t = t_first + (k - 1) / 3, plane = (k - 1) % 3;
      if (t >= T) {continue;}
      col = 1 + plane * T + t;
    }
    float acc = 0.0f;
    for (int i = lane; i < n; i += 32) {
      const float * p = parts + static_cast<size_t>(i) * stride;
      const float e = i < kMergeCached ? s_e[i] : expf(-(__ldg(p) - m) * inv_temp);
      acc = fmaf(__ldg(p + 1 + col), e, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {s_col[k] = acc;}
  }
  __syncthreads();
  if (tid < kMergeT && t_first + tid < T) {
    const int t = t_first + tid;
    const float ssum = s_col[0];
    const float wvx = s_col[1 + 3 * tid], wvy = s_col[2 + 3 * tid], wwz = s_col[3 + 3 * tid];
    if (!finalize) {
      dst[0] = m; dst[1] = ssum;
      dst[2 + t] = wvx; dst[2 + T + t] = wvy; dst[2 + 2 * T + t] = wwz;
    } else {
      // cs = W / sum, then applyControlSequenceConstraints (optimizer.cpp:237-249)
      float vx = wvx / ssum, wz = wwz / ssum, vy = bufs.cs[T + t];
      if (Pg->holonomic) {
        vy = wvy / ssum;
        vy = fminf(fmaxf(vy, -Pg->c_vy), Pg->c_vy);
      }
      vx = fminf(fmaxf(vx, Pg->c_vx_min), Pg->c_vx_max);
      wz = fminf(fmaxf(wz, -Pg->c_wz), Pg->c_wz);
      if (Pg->model == MPPI_MODEL_ACKERMANN) {   // motion_models.hpp:110-117
        const float r = Pg->min_turning_r;
        if (fabsf(vx) / fabsf(wz) < r) {
          const float sgn = wz > 0.0f ? 1.0f : (wz < 0.0f ? -1.0f : 0.0f);
          wz = sgn * fabsf(vx) / r;
        }
      }
      bufs.cs[t] = vx; bufs.cs[T + t] = vy; bufs.cs[2 * T + t] = wz;
      bufs.out[t] = vx; bufs.out[T + t] = vy; bufs.out[2 * T + t] = wz;
      if (host_res) {
        st_packet(host_res + t, __float_as_uint(vx), tag);
        st_packet(host_res + T + t, __float_as_uint(vy), tag);
        st_packet(host_res + 2 * T + t, __float_as_uint(wz), tag);
      }
    }
  }
  if (host_res && finalize && blockIdx.x == 0 && tid == 0) {
    // fail flag and furthest reached path point, published by the path-cost kernel in front of this one
    st_packet(host_res + 3 * T, __float_as_uint(bufs.out[3 * T]), tag);
    st_packet(host_res + 3 * T + 1, __float_as_uint(bufs.out[3 * T + 1]), tag);
  }
}

__global__ void __launch_bounds__(kUpdThreads) merge_finalize_kernel(
  const DevParams * __restrict__ Pg, const float * __restrict__ parts, int n, int stride, DevBuffers bufs, int finalize,
  float * __restrict__ dst, uint2 * host_res)
{
  // host_res: the tag is the packet epoch the path-cost kernel in front of this one advanced
  pdl_wait();
  merge_finalize_body(Pg, parts, n, stride, bufs, finalize, dst, host_res, host_res ? ld_volatile_u32(bufs.epoch) : 0u);
}

// K4p: exchange 2 over peer memory, fused with the merges on both sides of it.  Every block merges its columns of the
// rank's partial records (like merge_finalize_kernel) and PUSHES the merged slice into slot [rank] of every rank's
// mailbox; the last block to finish publishes the tag, waits for the tags of all ranks in its local mailbox, merges
// the nranks records and writes the new control sequence.  Every rank ends with the same sequence; no broadcast.
__global__ void __launch_bounds__(kUpdThreads) merge_exchange_finalize_kernel(
  const DevParams * __restrict__ Pg, const float * __restrict__ parts, int n, int stride, DevBuffers bufs)
{
  __shared__ float s_red[kUpdThreads / 32];
  __shared__ float s_col[3 * kMergeT + 1];
  __shared__ float s_e[kMergeCached];
  const PeerComm & pc = bufs.peer;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_wait();
  const int T = Pg->T;
  const float inv_temp = 1.0f / Pg->temperature;
  const unsigned tag = ld_volatile_u32(pc.seq) + 1u;
  // ---- local merge of this rank's partial records (identical to merge_finalize_kernel)
  float m = 3.402823466e+38f;
  for (int i = tid; i < n; i += kUpdThreads) {m = fminf(m, __ldg(parts + static_cast<size_t>(i) * stride));}
  m = warp_min(m);
  if (lane == 0) {s_red[warp] = m;}
  __syncthreads();
  m = s_red[0];
#pragma unroll
  for (int w = 1; w < kUpdThreads / 32; ++w) {m = fminf(m, s_red[w]);}
  for (int i = tid; i < min(n, kMergeCached); i += kUpdThreads) {
    s_e[i] = expf(-(__ldg(parts + static_cast<size_t>(i) * stride) - m) * inv_temp);
  }
  __syncthreads();
  const int t_first = blockIdx.x * kMergeT;
  for (int k = warp; k < 3 * kMergeT + 1; k += kUpdThreads / 32) {
    int col;
    if (k == 0) {
      col = 0;
    } else {
      const int t = t_first + (k - 1) / 3, plane = (k - 1) % 3;
      if (t >= T) {continue;}
      col = 1 + plane * T + t;
    }
    float acc = 0.0f;
    for (int i = lane; i < n; i += 32) {
      const float * p = parts + static_cast<size_t>(i) * stride;
      const float e = i < kMergeCached ? s_e[i] : expf(-(__ldg(p) - m) * inv_temp);
      acc = fmaf(__ldg(p + 1 + col), e, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {s_col[k] = acc;}
  }
  __syncthreads();
  // ---- push this block's merged values as packets into every rank's mailbox (remote stores over NVLink, slot = rank):
  //      record index 0 = m, 1 = s (block 0 only), 2 + plane * T + t = W
  if (tid < 3 * kMergeT + 1) {
    int idx = -1;
    if (tid == 0) {
      idx = blockIdx.x == 0 ? 1 : -1;
    } else {
      const int t = t_first + (tid - 1) / 3, plane = (tid - 1) % 3;
      if (t < T) {idx = 2 + plane * T + t;}
    }
    if (idx >= 0) {
      const unsigned bits = __float_as_uint(s_col[tid]);
#pragma unroll 1
      for (int r = 0; r < pc.nranks; ++r) {st_packet(pc.box[r] + kBoxX2 + pc.rank * kX2Stride + idx, bits, tag);}
    }
  } else if (tid == 32 && blockIdx.x == 0) {
    const unsigned bits = __float_as_uint(m);
#pragma unroll 1
    for (int r = 0; r < pc.nranks; ++r) {st_packet(pc.box[r] + kBoxX2 + pc.rank * kX2Stride, bits, tag);}
  }
  // ---- every block polls, in its LOCAL mailbox, the packets it needs from every rank: m, s and its own columns
  __shared__ float s_in[kMaxRanks][3 * kMergeT + 2];
  const uint2 * local = pc.box[pc.rank];
  constexpr int kNeed = 3 * kMergeT + 2;
  for (int i = tid; i < kNeed * pc.nranks; i += kUpdThreads) {
    const int r = i / kNeed, k = i - r * kNeed;   // k: 0 = m, 1 = s, 2.. = columns (t, plane)
    int idx = k;
    bool want = true;
    if (k >= 2) {
      const int t = t_first + (k - 2) / 3, plane = (k - 2) % 3;
      want = t < T;
      idx = 2 + plane * T + t;
    }
    unsigned bits = 0u;
    if (want && !poll_packet(local + kBoxX2 + r * kX2Stride + idx, tag, bits)) {raise_comm_error(bufs);}
    s_in[r][k] = __uint_as_float(bits);
  }
  __syncthreads();
  // ---- cross-rank merge of this block's time steps, cs = W / sum, applyControlSequenceConstraints (optimizer.cpp:237-249)
  if (tid < kMergeT && t_first + tid < T) {
    const int t = t_first + tid;
    float gm = 3.402823466e+38f;
    for (int r = 0; r < pc.nranks; ++r) {gm = fminf(gm, s_in[r][0]);}
    float ssum = 0.0f, wvx = 0.0f, wvy = 0.0f, wwz = 0.0f;
    for (int r = 0; r < pc.nranks; ++r) {
      const float e = expf(-(s_in[r][0] - gm) * inv_temp);
      ssum = fmaf(s_in[r][1], e, ssum);
      wvx = fmaf(s_in[r][2 + 3 * tid], e, wvx);
      wvy = fmaf(s_in[r][3 + 3 * tid], e, wvy);
      wwz = fmaf(s_in[r][4 + 3 * tid], e, wwz);
    }
    float vx = wvx / ssum, wz = wwz / ssum, vy = bufs.cs[T + t];
    if (Pg->holonomic) {
      vy = wvy / ssum;
      vy = fminf(fmaxf(vy, -Pg->c_vy), Pg->c_vy);
    }
    vx = fminf(fmaxf(vx, Pg->c_vx_min), Pg->c_vx_max);
    wz = fminf(fmaxf(wz, -Pg->c_wz), Pg->c_wz);
    if (Pg->model == MPPI_MODEL_ACKERMANN) {   // motion_models.hpp:110-117
      const float rr = Pg->min_turning_r;
      if (fabsf(vx) / fabsf(wz) < rr) {
        const float sgn = wz > 0.0f ? 1.0f : (wz < 0.0f ? -1.0f : 0.0f);
        wz = sgn * fabsf(vx) / rr;
      }
    }
    bufs.cs[t] = vx; bufs.cs[T + t] = vy; bufs.cs[2 * T + t] = wz;
    bufs.out[t] = vx; bufs.out[T + t] = vy; bufs.out[2 * T + t] = wz;
  }
  // ---- the last block to finish closes the round on this rank
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    if (atomicAdd(&bufs.st->ticket, 1u) == gridDim.x - 1) {
      bufs.st->ticket = 0u;
      bufs.out[3 * T + 5] = __uint_as_float(bufs.st->comm_error);
      __threadfence();
      *pc.seq = tag;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// small utility kernels
// ---------------------------------------------------------------------------------------------------
// time-major [T][B] -> row-major [B][T] (getGeneratedTrajectories / cell indices for the host; with the roles of T
// and B exchanged, [B][T] -> [T][B] for the noise of the stream layout).  The blocks of y stride over T: grid.y is capped
// at 65535, and a noise transpose puts the batch size there (transpose_grid).
template<typename V>
__global__ void transpose_tb_to_bt_kernel(const V * __restrict__ src, V * __restrict__ dst, int T, int B)
{
  __shared__ V tile[32][33];
  const int b0 = blockIdx.x * 32;
  for (int t0 = blockIdx.y * 32; t0 < T; t0 += gridDim.y * 32) {
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int t = t0 + i, b = b0 + threadIdx.x;
      if (t < T && b < B) {tile[i][threadIdx.x] = src[static_cast<size_t>(t) * B + b];}
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int b = b0 + i, t = t0 + threadIdx.x;
      if (t < T && b < B) {dst[static_cast<size_t>(b) * T + t] = tile[threadIdx.x][i];}
    }
    __syncthreads();
  }
}

// grid of transpose_tb_to_bt_kernel for a [T][B] source: B on x, T on y up to the 65535 blocks y allows
inline dim3 transpose_grid(int T, int B)
{
  const int ty = (T + 31) / 32;
  return dim3((B + 31) / 32, ty < 65535 ? ty : 65535);
}

// Optimizer::shiftControlSequence (optimizer.cpp:206-225): roll by -1, last = second to last
__global__ void shift_control_sequence_kernel(float * __restrict__ cs, int T, int holonomic)
{
  __shared__ float tmp[MPPI_MAX_TIME_STEPS];
  for (int plane = 0; plane < 3; ++plane) {
    if (plane == 1 && !holonomic) {continue;}
    float * v = cs + plane * T;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {tmp[t] = v[t];}
    __syncthreads();
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      // rolled[t] = old[t+1] (rolled[T-1] = old[0]); then rolled[T-1] = rolled[T-2] = old[T-1]
      v[t] = t < T - 1 ? tmp[t + 1] : (T >= 2 ? tmp[T - 1] : tmp[0]);
    }
    __syncthreads();
  }
}

// The tail of Optimizer::evalControl (optimizer.cpp:147-152) on the device, so that the control sequence never
// makes a host round trip between cycles: utils::savitskyGolayFilter (utils.hpp:442-605) with the 4-deep control
// history, getControlFromSequenceAsTwist (optimizer.cpp:396-410) and shiftControlSequence (:206-225).
// Skipped when the optimisation failed (fail_flag): the reference only reaches this code after fallback() returned
// false.  One thread per plane; the filter is inherently sequential (already-filtered neighbours are reused) and
// reproduces the reference's quirks: index num_sequences - 4 is never filtered, vy is filtered for every model.
// out layout: [0, 3T) control sequence after the tail, [3T] fail flag, [3T+1] furthest, [3T+2, 3T+5) command.
__global__ void eval_tail_kernel(float * __restrict__ cs, float * __restrict__ hist, float * __restrict__ out, int T, int holonomic, int shift)
{
  __shared__ float s[3][MPPI_MAX_TIME_STEPS];
  const int plane = threadIdx.x;   // 0 vx, 1 vy, 2 wz
  const bool failed = __float_as_int(out[3 * T]) != 0;
  if (plane < 3 && !failed) {
    float * v = s[plane];
    for (int t = 0; t < T; ++t) {v[t] = cs[plane * T + t];}
    out[3 * T + 2 + plane] = eval_tail_plane(v, hist, plane, T, holonomic, shift);
    for (int t = 0; t < T; ++t) {cs[plane * T + t] = v[t]; out[plane * T + t] = v[t];}
  } else if (plane < 3) {
    out[3 * T + 2 + plane] = 0.0f;
  }
}

// Optimizer::getOptimizedTrajectory (optimizer.cpp:345-360, :275-311): one trajectory from the mean controls
__global__ void optimized_trajectory_kernel(const float * __restrict__ cs, float * __restrict__ out_t3, int T, int holonomic,
  float dt, double pose_x, double pose_y, float yaw0)
{
  if (threadIdx.x != 0 || blockIdx.x != 0) {return;}
  float acc = 0.0f, accx = 0.0f, accy = 0.0f;
  for (int t = 0; t < T; ++t) {
    const float term = __fmul_rn(cs[2 * T + t], dt);
    acc = t == 0 ? term : __fadd_rn(acc, term);
    const float yaw = __fadd_rn(acc, yaw0);
    float sn, cn;
    // optimizer.cpp:294-299: cos/sin[0] of the initial yaw, cos/sin[t >= 1] of yaws[t] itself -- this overload has no
    // one-step lag, unlike the batch overload (:322-329)
    mppi_det_sincosf(t == 0 ? yaw0 : yaw, &sn, &cn);
    float dx = __fmul_rn(cs[t], cn), dy = __fmul_rn(cs[t], sn);
    if (holonomic) {
      dx = __fsub_rn(dx, __fmul_rn(cs[T + t], sn));
      dy = __fadd_rn(dy, __fmul_rn(cs[T + t], cn));
    }
    const float tx = __fmul_rn(dx, dt), ty = __fmul_rn(dy, dt);
    accx = t == 0 ? tx : __fadd_rn(accx, tx);
    accy = t == 0 ? ty : __fadd_rn(accy, ty);
    out_t3[3 * t] = static_cast<float>(pose_x + static_cast<double>(accx));
    out_t3[3 * t + 1] = static_cast<float>(pose_y + static_cast<double>(accy));
    out_t3[3 * t + 2] = yaw;
  }
}

// ---------------------------------------------------------------------------------------------------
// Multi-robot groups in the stream layout (BASELINE configs[4]): the four kernels of the large-batch path, launched
// ONCE for all robots of a group; the robot is the last grid dimension and its buffers come from the job table.
// Robots are independent problems (own record, costmap, noise, control sequence, state), so nothing else changes.
// Members may differ in batch_size and time_steps: each launch spans the largest member's extent in every grid dimension,
// and a block beyond its own member's extent returns before it touches anything (its partial records, its ticket).
// ---------------------------------------------------------------------------------------------------
// one robot of a group: where its record, costmap, buffers and pinned result packets are, and its launch extents (set by
// the host with the rules of the single-handle launches for this member's B and T)
struct __align__(16) FusedJob
{
  const DevParams * Pg;
  const uint8_t * cm;
  DevBuffers bufs;
  uint2 * host_res;
  int rollout_blocks;   // blocks of the rollout at the launch's block size
  int cost_blocks;      // path-cost blocks == partial minima (d_partials holds upd_blocks >= this many records)
  int ws_chunks;        // weighted-sums chunks == partial records the merge reads
  int merge_blocks;     // merge blocks (kMergeT steps each)
  int stride;           // floats per partial record, 3T + 2
};
static_assert(sizeof(FusedJob) % 16 == 0, "the job table is an array of 16-byte aligned records");

template<unsigned F, bool kExact>
__global__ void __launch_bounds__(kStreamThreads, MPPI_STREAM_MIN_BLOCKS) rollout_score_stream_batch_kernel(const FusedJob * __restrict__ jobs)
{
  const FusedJob & j = jobs[blockIdx.y];
  rollout_score_stream_body<F, kExact>(j.Pg, j.cm, j.bufs, j.rollout_blocks);
}

__global__ void __launch_bounds__(kUpdThreads, 5) path_costs_tm_batch_kernel(const FusedJob * __restrict__ jobs, int iteration)
{
  const FusedJob & j = jobs[blockIdx.y];
  if (static_cast<int>(blockIdx.x) >= j.cost_blocks) {return;}
  path_costs_tm_body(j.Pg, j.bufs, iteration, 0, static_cast<unsigned>(j.cost_blocks));
}

// blockIdx.y splits the member's 3T rows over gridDim.y groups: with a smaller T than the launch's, the trailing groups
// have no rows and only the first writes the record's [m, s]
__global__ void __launch_bounds__(kWsThreads) weighted_sums_tm_batch_kernel(const FusedJob * __restrict__ jobs)
{
  const FusedJob & j = jobs[blockIdx.z];
  if (static_cast<int>(blockIdx.x) >= j.ws_chunks) {return;}
  weighted_sums_tm_body(j.Pg, j.bufs);
}

// deliver = 0: an earlier iteration of a multi-iteration cycle, which only updates the control sequence
__global__ void __launch_bounds__(kUpdThreads) merge_finalize_batch_kernel(const FusedJob * __restrict__ jobs, unsigned tag, int deliver)
{
  const FusedJob & j = jobs[blockIdx.y];
  if (static_cast<int>(blockIdx.x) >= j.merge_blocks) {return;}
  merge_finalize_body(j.Pg, j.bufs.partials, j.ws_chunks, j.stride, j.bufs, 1, nullptr, deliver ? j.host_res : nullptr, tag);
}

// ---------------------------------------------------------------------------------------------------
// Path tables of a cycle whose costmap is device-resident (mppi_set_costmap_residency): build_params wrote the record
// without them, this kernel reads the map in place and writes valid[j], bits 0 / 1 of flags[f] (beside the PathAngle bit
// the host wrote) and follow_idx[f] into the device copy of the record, with build_params' own rules (mppi_device.cuh).
// One block, one thread per path point; both scans are integer, so the tables are the host's bit for bit.  A record
// without a device map (cm_dev == null: a host-mode member of a group) is left alone.
// ---------------------------------------------------------------------------------------------------
constexpr int kTablesThreads = MPPI_MAX_PATH_POINTS;
static_assert(kTablesThreads == 32 * 32, "the scans below combine 32 warps of 32 lanes");

__device__ __forceinline__ void path_tables_body(DevParams * P)
{
  __shared__ uint16_t s_inv[kTablesThreads + 1];   // invalid points among [0, j)
  __shared__ int s_next[kTablesThreads + 1];        // first valid index >= j, N if none
  __shared__ int s_warp[2][32];
  const uint8_t * cm = P->cm_dev;
  if (cm == nullptr) {return;}
  const int N = P->N, n16 = ((N + 15) / 16) * 16;
  const int j = threadIdx.x, lane = j & 31, warp = j >> 5;
  const float * path = reinterpret_cast<const float *>(P + 1);
  uint8_t * valid = reinterpret_cast<uint8_t *>(const_cast<float *>(path) + 4 * N);
  uint8_t * flags = valid + n16;
  uint16_t * follow = reinterpret_cast<uint16_t *>(valid + 2 * n16);
  bool ok = false;
  if (j < N - 1) {
    ok = path_point_valid(cm, P->size_x, P->size_y, P->res, P->ox, P->oy, P->track_unknown,
      static_cast<double>(path[P->off_path_x + j]), static_cast<double>(path[P->off_path_y + j]));
  }
  // inclusive prefix count of the invalid points (the last point counts: it is never valid) and suffix minimum of the
  // valid indices, per warp with shuffles, then across the 32 warp totals
  int inv = (j < N && !ok) ? 1 : 0;
  int nxt = (j < N && ok) ? j : N;
  for (int o = 1; o < 32; o <<= 1) {
    const int a = __shfl_up_sync(0xffffffffu, inv, o), b = __shfl_down_sync(0xffffffffu, nxt, o);
    if (lane >= o) {inv += a;}
    if (lane + o < 32) {nxt = min(nxt, b);}
  }
  if (lane == 31) {s_warp[0][warp] = inv;}
  if (lane == 0) {s_warp[1][warp] = nxt;}
  __syncthreads();
  if (warp == 0) {
    int wi = s_warp[0][lane], wn = s_warp[1][lane];
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, wi, o), b = __shfl_down_sync(0xffffffffu, wn, o);
      if (lane >= o) {wi += a;}
      if (lane + o < 32) {wn = min(wn, b);}
    }
    s_warp[0][lane] = wi;
    s_warp[1][lane] = wn;
  }
  __syncthreads();
  if (warp > 0) {inv += s_warp[0][warp - 1];}
  if (warp < 31) {nxt = min(nxt, s_warp[1][warp + 1]);}
  s_inv[j + 1] = static_cast<uint16_t>(inv);
  if (j == 0) {s_inv[0] = 0;}
  s_next[j] = nxt;
  __syncthreads();
  if (j < N) {
    valid[j] = ok ? 1 : 0;
    follow[j] = static_cast<uint16_t>(path_follow_index(j, P->follow_offset, N, s_next));
    flags[j] = static_cast<uint8_t>((flags[j] & 4u) | path_align_flag_bits(*P, j, s_inv));
  }
}

__global__ void __launch_bounds__(kTablesThreads) path_tables_kernel(DevParams * P)
{
  path_tables_body(P);
}

// a chunk of a robot group: member = blockIdx.y
__global__ void __launch_bounds__(kTablesThreads) path_tables_batch_kernel(const FusedJob * __restrict__ jobs)
{
  path_tables_body(const_cast<DevParams *>(jobs[blockIdx.y].Pg));
}

// ---------------------------------------------------------------------------------------------------
// Cycle records of a robot group built on the device from inputs in device memory (mppi_optimize_group_device).
// The host builds each member's TEMPLATE once per configuration change: a record made by build_params itself (constraints,
// gamma terms, critic table, footprint, ObstaclesCritic LUTs, map geometry and circumscribed cost) followed by the
// thresholds below.  Per cycle, record_batch_kernel copies the template into the member's slice of the group arena and
// completes everything build_params derives from the cycle inputs, with build_params' arithmetic: the pose and speed
// fields, the path tail (x, y, yaw, the arc-length prefix D as a sequential fp32 sum), closest_path_pt, the path spacing
// bounds, the goal gates (within_tolerance & co, mppi_device.cuh), PathAngle's gate per index and the fields derived from
// the gates.  path_tables_batch_kernel runs right behind it and makes the costmap-dependent tables.
// ---------------------------------------------------------------------------------------------------
struct RecordGates
{
  double angle_cos_max;                      // cos(max_angle_to_furthest), host libm (PathAngle's fast test)
  float goal_thr, goal_angle_thr, forward_thr, follow_thr, align_thr, legacy_thr, angle_thr;   // threshold_to_consider
  float cost_near, obst_near;                // near_goal_distance of CostCritic / ObstaclesCritic
  float angle_max;                           // max_angle_to_furthest
  int goal_en, goal_angle_en, forward_en, twirl_en, follow_en, align_en, legacy_en, angle_en;   // in the list and enabled
  int has_cost, has_obst;                    // in the list
  int angle_fast;                            // the fast test applies (forward_preference, 1e-3 < max < 3.1)
  int want_traj;                             // MPPI_WANT_TRAJECTORIES
};
constexpr int kTemplateStride = ((static_cast<int>(sizeof(DevParams) + sizeof(RecordGates)) + 15) / 16) * 16;
static_assert(sizeof(DevParams) % 8 == 0, "the template is copied in 8-byte words");

constexpr int kRecordThreads = 256;
// value of a member's status packet (host_res[3T + 8]): the PathAngle band hits of the cycle, or this bit for a path_size
// outside [1, min(MPPI_MAX_PATH_POINTS, path_stride)] (the member's launches are then cancelled, nothing of it changes)
constexpr unsigned kRecordBadPath = 0x80000000u;

// posePointAngle (utils.hpp:417-434) with the device's atan2f: used only inside PathAngle's undecided band
__device__ __noinline__ float pose_point_angle_dev(float pose_xf, float pose_yf, float pose_yawf, float gx, float gy, bool forward_preference)
{
  const float yaw = atan2f(__fsub_rn(gy, pose_yf), __fsub_rn(gx, pose_xf));
  const double a = fabs(normalize_angle_d(__dsub_rn(static_cast<double>(pose_yawf), static_cast<double>(yaw))));
  if (forward_preference) {return static_cast<float>(a);}
  const double back = normalize_angle_d(__dadd_rn(static_cast<double>(pose_yawf), 3.14159265358979323846));
  return static_cast<float>(fmin(a, fabs(normalize_angle_d(__dsub_rn(back, static_cast<double>(yaw))))));
}

// noise_jobs / noise_index: the group's regenerate_noises table and each member's entry in it (-1: none)
__global__ void __launch_bounds__(kRecordThreads) record_batch_kernel(FusedJob * __restrict__ jobs, const char * __restrict__ templates,
  mppi_group_inputs in, int row0, unsigned tag, NoiseJob * __restrict__ noise_jobs, const int * __restrict__ noise_index)
{
  __shared__ float s_seg[MPPI_MAX_PATH_POINTS];          // fp32 length of segment i - 1 -> i (D)
  __shared__ double s_segd[MPPI_MAX_PATH_POINTS];        // fp64 length of segment j -> j + 1 (path spacing)
  __shared__ uint8_t s_gate[MPPI_MAX_PATH_POINTS];       // PathAngle gate per candidate target index
  __shared__ unsigned long long s_closest, s_hmax;
  __shared__ unsigned s_band, s_open;
  __shared__ double s_len;
  FusedJob & job = jobs[blockIdx.y];
  DevParams * P = const_cast<DevParams *>(job.Pg);
  const int row = row0 + static_cast<int>(blockIdx.y), tid = threadIdx.x;
  const DevParams * tp = reinterpret_cast<const DevParams *>(templates + static_cast<size_t>(row) * kTemplateStride);
  const RecordGates & g = *reinterpret_cast<const RecordGates *>(tp + 1);
  const int N = in.path_size[row];
  if (N < 1 || N > MPPI_MAX_PATH_POINTS || N > in.path_stride) {
    if (tid == 0) {
      // cancel the member's launches (their blocks return at once) and its noise redraws (no items; the host restores the
      // entry and the epoch), keep the path tables away from its stale record
      job.rollout_blocks = 0; job.cost_blocks = 0; job.ws_chunks = 0; job.merge_blocks = 0;
      if (noise_index[row] >= 0) {noise_jobs[noise_index[row]].B = 0;}
      P->cm_dev = nullptr;
      st_packet(job.host_res + 3 * tp->T + 8, kRecordBadPath, tag);
    }
    return;
  }
  {
    const unsigned long long * src = reinterpret_cast<const unsigned long long *>(tp);
    unsigned long long * dst = reinterpret_cast<unsigned long long *>(P);
    for (int i = tid; i < static_cast<int>(sizeof(DevParams) / 8); i += kRecordThreads) {dst[i] = src[i];}
  }
  if (tid == 0) {s_closest = (static_cast<unsigned long long>(__float_as_uint(3.402823466e+38f)) << 32); s_hmax = 0ull; s_band = 0u; s_open = 0u;}
  const double * st = in.state + 8 * static_cast<size_t>(row);
  const double rx = st[0], ry = st[1], ryaw = st[2], gx = st[6], gy = st[7];
  const float * px = in.path + static_cast<size_t>(row) * 3 * in.path_stride;
  const float * py = px + in.path_stride, * pyaw = py + in.path_stride;
  const float yaw0 = static_cast<float>(ryaw);
  float sin0, cos0;
  mppi_det_sincosf(yaw0, &sin0, &cos0);
  const float svx = static_cast<float>(st[3]), svy = static_cast<float>(st[4]);
  // trajectory 0's first pose (build_params: the rollout's own arithmetic)
  float x00, y00;
  {
    const bool hol = tp->holonomic != 0;
    const float vx0 = svx, vy0 = hol ? svy : 0.0f;
    float dx = __fmul_rn(vx0, cos0), dy = __fmul_rn(vx0, sin0);
    if (hol) {dx = __fsub_rn(dx, __fmul_rn(vy0, sin0)); dy = __fadd_rn(dy, __fmul_rn(vy0, cos0));}
    x00 = static_cast<float>(__dadd_rn(rx, static_cast<double>(__fmul_rn(dx, tp->dt))));
    y00 = static_cast<float>(__dadd_rn(ry, static_cast<double>(__fmul_rn(dy, tp->dt))));
  }
  const bool angle_on = g.angle_en && !within_tolerance(g.angle_thr, rx, ry, gx, gy);
  const float pose_xf = static_cast<float>(rx), pose_yf = static_cast<float>(ry);
  double sh = 0.0, ch = 1.0;
  if (angle_on && g.angle_fast) {sincos(static_cast<double>(yaw0), &sh, &ch);}
  const int n16 = ((N + 15) / 16) * 16;
  float * tail = reinterpret_cast<float *>(P + 1);
  uint8_t * valid = reinterpret_cast<uint8_t *>(tail + 4 * N);
  uint8_t * flags = valid + n16;
  __syncthreads();   // the template is in place, the shared accumulators are set
  for (int i = tid; i < 2 * n16 + 2 * N; i += kRecordThreads) {valid[i] = 0;}
  const int open_from = max(0, min(tp->angle_offset, N - 1));
  unsigned long long best = ~0ull, hmax = 0ull;
  unsigned band = 0u, open_any = 0u;
  for (int j = tid; j < N; j += kRecordThreads) {
    const float xj = px[j], yj = py[j];
    tail[j] = xj; tail[N + j] = yj; tail[2 * N + j] = pyaw[j];
    if (j > 0) {
      const float dx = __fsub_rn(xj, px[j - 1]), dy = __fsub_rn(yj, py[j - 1]);
      s_seg[j] = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
    }
    if (j + 1 < N) {
      const double sx = __dsub_rn(static_cast<double>(px[j + 1]), static_cast<double>(xj));
      const double sy = __dsub_rn(static_cast<double>(py[j + 1]), static_cast<double>(yj));
      const double seg = __dsqrt_rn(__dadd_rn(__dmul_rn(sx, sx), __dmul_rn(sy, sy)));
      s_segd[j] = seg;
      if (seg >= 0.0) {hmax = max(hmax, static_cast<unsigned long long>(__double_as_longlong(seg)));}   // NaN is skipped, as std::max does
    }
    {
      const float dx = __fsub_rn(xj, x00), dy = __fsub_rn(yj, y00);
      const float d = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
      if (d < 3.402823466e+38f) {best = min(best, (static_cast<unsigned long long>(__float_as_uint(d)) << 32) | static_cast<unsigned>(j));}
    }
    bool open = false;
    if (angle_on) {
      int decided = g.angle_fast ? path_angle_fast_gate(xj, yj, pose_xf, pose_yf, ch, sh, g.angle_cos_max) : -1;
      if (decided < 0) {
        // the point under the robot is no band decision: atan2f(+0, +0) = +0 on either side
        band += (__fsub_rn(xj, pose_xf) != 0.0f || __fsub_rn(yj, pose_yf) != 0.0f) ? 1u : 0u;
        decided = pose_point_angle_dev(pose_xf, pose_yf, yaw0, xj, yj, tp->angle_forward_pref != 0) < g.angle_max ? 0 : 1;
      }
      open = decided == 1;
    }
    s_gate[j] = open ? 1 : 0;
    if (open && j >= open_from) {open_any = 1u;}
  }
  if (best != ~0ull) {atomicMin(&s_closest, best);}
  if (hmax != 0ull) {atomicMax(&s_hmax, hmax);}
  if (band) {atomicAdd(&s_band, band);}
  if (open_any) {s_open = 1u;}
  __syncthreads();
  if (tid == 0) {
    // arc-length prefix (path_align_critic.cpp:83-90): a sequential fp32 sum in index order, as build_params makes it
    float * D = tail + 3 * N;
    float acc = 0.0f;
    D[0] = 0.0f;
    for (int i = 1; i < N; ++i) {acc = __fadd_rn(acc, s_seg[i]); D[i] = acc;}
  } else if (tid == 32) {
    double len = 0.0;
    for (int j = 0; j + 1 < N; ++j) {len = __dadd_rn(len, s_segd[j]);}
    s_len = len;
  }
  for (int f = tid; f < N; f += kRecordThreads) {
    if (s_gate[min(f + tp->angle_offset, N - 1)]) {flags[f] = 4u;}
  }
  __syncthreads();
  if (tid != 0) {return;}
  DevParams & p = *P;
  p.pose_x = rx; p.pose_y = ry;
  p.yaw0 = yaw0; p.sin0 = sin0; p.cos0 = cos0;
  p.speed_vx = svx; p.speed_vy = svy; p.speed_wz = static_cast<float>(st[5]);
  p.goal_x = gx; p.goal_y = gy;
  p.N = N;
  p.goal_yaw = pyaw[N - 1];
  p.off_path_x = 0; p.off_path_y = N; p.off_path_yaw = 2 * N; p.off_path_D = 3 * N;
  p.cm_dev = job.cm;
  p.closest_path_pt = s_closest == (static_cast<unsigned long long>(__float_as_uint(3.402823466e+38f)) << 32) ? 0 :
    static_cast<int>(s_closest & 0xFFFFFFFFull);
  {
    const double hm = __longlong_as_double(static_cast<long long>(s_hmax)), len = s_len;
    p.path_hmax_inv = (hm > 0.0 && isfinite(hm)) ? static_cast<float>(__ddiv_rn(1.0, __dmul_rn(hm, 1.00001))) : 0.0f;
    p.path_hmean_inv = (len > 0.0 && isfinite(len)) ? static_cast<float>(__ddiv_rn(static_cast<double>(N - 1), len)) : 0.0f;
  }
  // the gates (build_params, in its order)
  if (g.has_cost) {p.cost_near_goal = within_tolerance(g.cost_near, rx, ry, gx, gy) ? 1 : 0;}
  if (g.has_obst) {p.obst_near_goal = within_tolerance(g.obst_near, rx, ry, gx, gy) ? 1 : 0;}
  p.goal.on = g.goal_en && within_tolerance(g.goal_thr, rx, ry, gx, gy);
  p.goal_angle.on = g.goal_angle_en && within_tolerance(g.goal_angle_thr, rx, ry, gx, gy);
  p.forward.on = g.forward_en && !within_tolerance(g.forward_thr, rx, ry, gx, gy);
  p.twirl.on = g.twirl_en && !within_checker_tolerance(in.goal_checker_xy_tolerance[row], rx, ry, gx, gy);
  p.follow.on = g.follow_en && N >= 2 && !within_tolerance(g.follow_thr, rx, ry, gx, gy);
  p.align.on = g.align_en && !within_tolerance(g.align_thr, rx, ry, gx, gy);
  p.legacy.on = g.legacy_en && !within_tolerance(g.legacy_thr, rx, ry, gx, gy);
  p.angle.on = angle_on;
  if (p.align.on || p.legacy.on) {
    p.sample_step = p.align.on ? p.align_step : p.legacy_step;
    p.n_samples = (p.T + p.sample_step - 1) / p.sample_step;
    p.sample_yaw = (p.align.on && p.align_use_yaw) || (p.legacy.on && p.legacy_use_yaw);
  } else {
    p.sample_step = 0; p.n_samples = 0; p.sample_yaw = 0;
  }
  p.obstacle_q[0] = p.obstacle_q[1] = -1;
  p.first_path_q = -1;
  int nob = 0;
  for (int q = 0; q < p.n_critics; ++q) {
    const int kind = p.kind_of[q];
    const bool obstacle_like = (kind == MPPI_CRITIC_COST && p.cost.on) || (kind == MPPI_CRITIC_OBSTACLES && p.obst.on);
    if (obstacle_like && nob < 2) {p.obstacle_q[nob++] = q;}
    const bool path_like = (kind == MPPI_CRITIC_PATH_FOLLOW && p.follow.on) || (kind == MPPI_CRITIC_PATH_ANGLE && p.angle.on) ||
      (kind == MPPI_CRITIC_PATH_ALIGN && p.align.on) || (kind == MPPI_CRITIC_PATH_ALIGN_LEGACY && p.legacy.on);
    if (path_like && p.first_path_q < 0) {p.first_path_q = q;}
    int on = 0;
    switch (kind) {
      case MPPI_CRITIC_PATH_FOLLOW: on = p.follow.on ? 2 : 0; break;
      case MPPI_CRITIC_PATH_ALIGN: on = p.align.on ? 3 : 0; break;
      case MPPI_CRITIC_PATH_ALIGN_LEGACY: on = p.legacy.on ? 4 : 0; break;
      case MPPI_CRITIC_PATH_ANGLE: on = p.angle.on ? 5 : 0; break;
      case MPPI_CRITIC_GOAL: on = p.goal.on; break;
      case MPPI_CRITIC_GOAL_ANGLE: on = p.goal_angle.on; break;
      case MPPI_CRITIC_PREFER_FORWARD: on = p.forward.on; break;
      case MPPI_CRITIC_TWIRLING: on = p.twirl.on; break;
      default: on = p.src_base[q]; break;   // not gated per cycle: the template's
    }
    p.src_base[q] = static_cast<unsigned char>(on);
  }
  p.spill_traj = (g.want_traj || s_open) ? 1 : 0;
  __threadfence_system();
  st_packet(job.host_res + 3 * p.T + 8, s_band, tag);
}

}  // namespace mppi
