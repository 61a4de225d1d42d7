// mppi_device.cuh -- device-side data layout and helpers shared by the kernels.
//
// HBM layout (all owned by one mppi_handle, allocated once at create):
//   noise_vx/vy/wz   float [B][T] row-major   the reference's layout (models/state.hpp), so that injected
//                                              noise is a plain copy; read once per kernel, coalesced
//   costmap          uint8 [size_y][size_x]    uploaded once per cycle with one async copy, or read in place from
//                                              the caller's device memory (mppi_set_costmap_residency)
//   DevParams + path one packed record         uploaded once per cycle with one async copy
//   crit_rows        float [R][B]              per-critic contribution rows + 3 gamma rows (plane-major =
//                                              coalesced for lane == trajectory)
//   samples / ends   float [K][B], [2][B]      every trajectory_point_step-th pose for PathAlign, end pose
//   spill x/y/yaw    float [T][B] time-major   only when PathAngle may fire or trajectories are requested
//   costs            float [B]                 persists across iteration_count iterations (quirk R20)
//   partials         float [blocks][3T+2]      online-softmax partials merged by the last block
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <cmath>

#include "../../include/mppi_b200.h"
#include "../../include/mppi_det_math.h"

namespace mppi
{

// Optional phase trace (build with -DMPPI_TRACE; tuning aid, not part of the product build): SM clock at phase
// boundaries as seen by thread 0 of block 0, read back with mppi_debug_get_trace().
#ifdef MPPI_TRACE
__device__ long long g_trace[64];
#define MPPI_TRACE_AT(i) do {if (blockIdx.x == 0 && threadIdx.x == 0 && threadIdx.y == 0) {g_trace[i] = clock64();}} while (0)
#else
#define MPPI_TRACE_AT(i) do {} while (0)
#endif

constexpr int kTile = 32;          // trajectories per tile == warp width (lane = trajectory)
constexpr int kPad = 33;           // smem row pitch of the time-major tile [T][33]: conflict-free both ways
constexpr int kMaxCritics = MPPI_MAX_CRITICS;
constexpr int kGammaRows = 3;      // gamma-term rows stored after the critic rows
constexpr unsigned kUnset = 0xFFFFFFFFu;

constexpr unsigned char NO_INFORMATION = 255;
constexpr unsigned char LETHAL_OBSTACLE = 254;
constexpr unsigned char INSCRIBED_INFLATED_OBSTACLE = 253;

struct CriticCommon
{
  int idx;            // position in the critics list, -1 when the kind is absent
  int on;             // enabled && this cycle's host-side gate (withinPositionGoalTolerance & co) lets it run
  unsigned power;
  float weight;
};

// One record per cycle.  Scalars the host can decide (goal-distance gates, PathAngle gate per candidate
// index, arc-length prefix of the path) are decided on the host with the same libm the oracle uses, so
// every discrete decision taken on the device is a pure function of bit-exact inputs.
struct DevParams
{
  int B, T, N, n_critics;
  int holonomic, model;
  int mode;                 // 0 rollout from noise, 1 injected state (integrate), 2 injected state + trajectories
  float dt, min_turning_r;
  float yaw0, cos0, sin0;
  float speed_vx, speed_vy, speed_wz;
  float goal_yaw;
  float temperature;
  float gamma_vx, gamma_vy, gamma_wz;        // gamma / std^2
  float c_vx_max, c_vx_min, c_vy, c_wz;      // current (speed-limited) constraints
  unsigned size_x, size_y;
  int track_unknown;
  unsigned preset_furthest;                  // score mode: caller-provided furthest point, kUnset otherwise
  double pose_x, pose_y;
  double goal_x, goal_y;
  double res, ox, oy;
  int kind_of[kMaxCritics];                  // list order -> kind
  // per kind
  CriticCommon constraint; float max_vel, min_vel;
  CriticCommon cost; int cost_fp; float cost_critical, cost_collision; int cost_near_goal; float cost_possibly_inscribed;
  CriticCommon goal;
  CriticCommon goal_angle;
  CriticCommon obst; int obst_fp; float obst_collision, obst_critical_w, obst_repulsion_w; int obst_near_goal;
  float obst_possibly_inscribed; int obst_repulsion_enabled;
  CriticCommon align; int align_offset, align_step, align_use_yaw; float align_max_ratio;
  CriticCommon legacy; int legacy_offset, legacy_step, legacy_use_yaw; float legacy_max_ratio;
  CriticCommon angle; int angle_offset; int angle_reversing, angle_forward_pref;
  CriticCommon follow; int follow_offset;
  CriticCommon forward;
  CriticCommon twirl;
  CriticCommon deadband; float db_vx, db_vy, db_wz;
  // spills
  int sample_step, n_samples, sample_yaw;    // PathAlign samples: p = 0, step, 2 step ... < T
  int spill_traj;                            // write x,y,yaw time-major (PathAngle may fire / requested)
  int want_cells;
  int vis_b_step, vis_t_step, vis_nb;        // visualiser feed: every vis_b_step-th trajectory x every vis_t_step-th step (0: off)
  int need_furthest;                         // some path critic may ask for the furthest reached path point
  int noise_tm;                              // noise planes are stored time-major [T][B] (stream layout) instead of [B][T]
  // offsets (in floats) of the path arrays that follow this struct in the same buffer
  int off_path_x, off_path_y, off_path_yaw, off_path_D;
  // tables behind the path arrays, made by build_params (host map) or path_tables_kernel (device map; bit 2 of the
  // flags always by the host): valid[n16] (utils::findPathCosts, utils.hpp:361-394), flags[n16] and follow_idx[N]
  // (uint16), the last two indexed by the furthest reached path point: bit 0 PathAlign gate, bit 1 PathAlignLegacy gate,
  // bit 2 PathAngle gate; PathFollow's target index
  int obstacle_q[2];                         // list positions of the enabled obstacle-type critics (Cost / Obstacles), -1 if none
  int first_path_q;                          // list position of the first enabled path critic, -1 if none
  int closest_path_pt;                       // utils::findPathTrajectoryInitialPoint (utils.hpp:327-344), host decided
  int want_critic_rows;                      // per-critic rows are read back by the caller: keep them fully defined
  int fp_n;
  float cell_oxf, cell_oyf, cell_invf;       // fp32 filter of worldToMap (world_to_cell_fast): fl32(ox), fl32(oy), fl32(1/res)
  float cell_eps_x, cell_eps_y;              // and its error bounds in cells
  // furthest-point search of the stream kernel (utils.hpp:292-319 restated as a scan that skips): 1 / (longest path
  // segment, rounded up) bounds how fast the distance to the path can fall from one point to the next; (N - 1) / length
  // places the first guess.  Zero: no skipping / no guess.
  float path_hmax_inv, path_hmean_inv;
  // where the term of list position q comes from when the critic runs (fused kernel): 0 nothing (absent / disabled / gated
  // off by the host), 1 K2's row, 2 PathFollow, 3 PathAlign, 4 PathAlignLegacy, 5 PathAngle
  unsigned char src_base[kMaxCritics];
  // ---- everything above is the "hot" part every CTA copies into shared memory (kHotBytes) ----
  double fp_x[MPPI_MAX_FOOTPRINT], fp_y[MPPI_MAX_FOOTPRINT];   // footprint polygon
  // obstacle-critic look-up tables indexed by the byte cost: [0] point cost, [1] footprint cost
  float obst_lut_crit[2][256];               // (d < margin) ? margin - d : 0
  float obst_lut_rep[2][256];                // (d < margin) ? 0 : inflation_radius - d
  // the caller's device-resident costmap of this cycle (mppi_set_costmap_residency), null for a host map.  The kDevMap
  // instances of the rollout kernels read their map from here, so that a captured graph follows the pointer of every cycle.
  const uint8_t * cm_dev;
};
constexpr int kHotBytes = (static_cast<int>(offsetof(DevParams, fp_x)) + 15) & ~15;

// ---- the costmap-dependent path tables, one definition for build_params (host map) and path_tables_kernel (device
//      map).  Integer logic and IEEE sub / div only (no product to contract), so both sides produce the same bits.
// utils::findPathCosts (utils.hpp:361-394): the path point (wx, wy) is valid unless worldToMap fails (fp64) or its cell is
// lethal, inscribed, or unknown while unknown space is not tracked
__host__ __device__ inline bool path_point_valid(const uint8_t * cells, unsigned size_x, unsigned size_y, double res, double ox,
  double oy, int track_unknown, double wx, double wy)
{
  if (wx < ox || wy < oy) {return false;}
  const double qx = (wx - ox) / res, qy = (wy - oy) / res;
  if (!(qx < static_cast<double>(size_x) && qy < static_cast<double>(size_y))) {return false;}
  const unsigned mx = static_cast<unsigned>(qx), my = static_cast<unsigned>(qy);
  if (!(mx < size_x && my < size_y)) {return false;}
  const int c = cells[static_cast<size_t>(my) * size_x + mx];
  return !(c == LETHAL_OBSTACLE || c == INSCRIBED_INFLATED_OBSTACLE || (c == NO_INFORMATION && !track_unknown));
}
// PathAlign's occupancy gate for the furthest reached point f (path_align_critic.cpp:56-72); invalid_before[j] = number of
// invalid points among [0, j).  The reference bails out of its counting loop as soon as ctr / range > ratio with ctr > 2;
// the count only grows and the range is fixed, so the final count decides.
__host__ __device__ inline bool path_align_gate(int f, int offset, float max_ratio, int closest, const uint16_t * invalid_before)
{
  if (f < offset) {return false;}
  const float range = static_cast<float>(static_cast<long long>(f) - closest);
  unsigned invalid_ctr = 0;
  if (f > closest) {invalid_ctr = static_cast<unsigned>(invalid_before[f]) - static_cast<unsigned>(invalid_before[closest]);}
  return !(invalid_ctr > 2 && static_cast<float>(invalid_ctr) / range > max_ratio);
}
// bits 0 (PathAlign) and 1 (PathAlignLegacy) of the flag byte of furthest point f
__host__ __device__ inline unsigned path_align_flag_bits(const DevParams & p, int f, const uint16_t * invalid_before)
{
  unsigned fl = 0;
  if (path_align_gate(f, p.align_offset, p.align_max_ratio, p.closest_path_pt, invalid_before) && f > 0) {fl |= 1u;}
  if (path_align_gate(f, p.legacy_offset, p.legacy_max_ratio, p.closest_path_pt, invalid_before) && (p.N - 1) >= 1) {fl |= 2u;}
  return fl;
}
// PathFollow's target for furthest point f (path_follow_critic.cpp:45-58); next_valid[i] = first valid index >= i
__host__ __device__ inline int path_follow_index(int f, int offset, int N, const int * next_valid)
{
  const int path_size = N - 1;
  int fidx = f + offset < path_size ? f + offset : path_size;
  if (fidx < path_size - 1) {fidx = next_valid[fidx] < path_size - 1 ? next_valid[fidx] : path_size - 1;}
  return fidx > 0 ? fidx : 0;
}
constexpr int kHotFloats = kHotBytes / 4;

// ---- the per-cycle goal gates, one definition for build_params (host inputs) and record_batch_kernel (device inputs).
//      IEEE mul / add only, never contracted (the host pass is built with -ffp-contract=off), so both sides decide alike.
#if defined(__CUDA_ARCH__)
#define MPPI_DADD(a, b) __dadd_rn((a), (b))
#else
#define MPPI_DADD(a, b) ((a) + (b))
#endif
// utils::withinPositionGoalTolerance(float, ...) utils.hpp:233-249 (std::pow(d, 2) is d * d, exactly)
__host__ __device__ inline bool within_tolerance(float pose_tolerance, double rx, double ry, double gx, double gy)
{
  const double dx = gx - rx, dy = gy - ry;
  const double dist_sq = MPPI_DADD(MPPI_DMUL(dx, dx), MPPI_DMUL(dy, dy));
  const float pose_tolerance_sq = MPPI_FMUL(pose_tolerance, pose_tolerance);
  return dist_sq < pose_tolerance_sq;
}
// utils::withinPositionGoalTolerance(GoalChecker*, ...) utils.hpp:201-224
__host__ __device__ inline bool within_checker_tolerance(double tol, double rx, double ry, double gx, double gy)
{
  if (tol >= 0.0) {
    const double dx = rx - gx, dy = ry - gy;
    if (MPPI_DADD(MPPI_DMUL(dx, dx), MPPI_DMUL(dy, dy)) < MPPI_DMUL(tol, tol)) {return true;}
  }
  return false;
}
// PathAngle's gate for the path point (gx, gy) with forward_preference (path_angle_critic.cpp:79-83): the angle A in
// [0, pi] between the heading (cos ch, sin sh) and the direction to the point is below max (cos max = ct) iff
// cos A > ct.  Decided from a dot product wherever that is further than 1e-5 from the threshold (atan2f, the float roundings
// of the reference and the rounding of A to float move cos A by < 1e-6): 1 open, 0 closed, -1 undecided (the caller
// evaluates posePointAngle itself).
__host__ __device__ inline int path_angle_fast_gate(float gx, float gy, float pose_xf, float pose_yf, double ch, double sh, double ct)
{
  const double dxj = static_cast<double>(MPPI_FSUB(gx, pose_xf)), dyj = static_cast<double>(MPPI_FSUB(gy, pose_yf));
  const double dd = MPPI_DADD(MPPI_DMUL(dxj, dxj), MPPI_DMUL(dyj, dyj));
  if (dd > 1.0e-12) {
#if defined(__CUDA_ARCH__)
    const double c = __ddiv_rn(MPPI_DADD(MPPI_DMUL(dxj, ch), MPPI_DMUL(dyj, sh)), __dsqrt_rn(dd));
#else
    const double c = (dxj * ch + dyj * sh) / std::sqrt(dd);
#endif
    if (c < ct - 1.0e-5) {return 1;}
    if (c > ct + 1.0e-5) {return 0;}
  }
  return -1;
}

// cooperative copy of the hot part of the record into shared memory (16-byte vectors, coalesced)
__device__ __forceinline__ void load_hot_params(float * s_hot, const DevParams * __restrict__ P, int tid, int nthreads)
{
  const float4 * src = reinterpret_cast<const float4 *>(P);
  float4 * dst = reinterpret_cast<float4 *>(s_hot);
  for (int i = tid; i < kHotBytes / 16; i += nthreads) {dst[i] = __ldg(src + i);}
}

// ---------------------------------------------------------------------------------------------------
// Peer-memory exchange between the ranks of a sharded problem (one process per GPU, NVLink / NVSwitch).
// Every rank owns a small MAILBOX in its own HBM and maps the mailboxes of all peers (CUDA IPC).  Data travels as
// 8-byte PACKETS {value, tag}: one aligned 8-byte store is delivered whole, so a packet whose tag equals the tag of
// the current round IS its own arrival flag (the "LL" idea of NCCL's low-latency protocol).  A rank pushes its
// contribution into slot [its rank] of every mailbox with plain remote stores; consumers spin on packets in their
// LOCAL memory.  No fences, no separate flags, no NCCL call, no extra kernel, no host involvement: one one-way NVLink
// latency per exchange.  Exchange 1 rides at the start of K3, exchange 2 inside the merge kernel (SURVEY 8e).
// Spins are bounded: a peer that never arrives raises comm_error instead of hanging.  Tags are the round counter
// (*seq + 1, 32 bit, never reset): a stale packet of an older round can never match.
//   mailbox packets:  x1 [kMaxRanks][kX1Words]   words 0..16 = furthest candidate + survivor flags
//                     x2 [kMaxRanks][kX2Stride]  (m, s, W[3T]) softmax record of the rank
// ---------------------------------------------------------------------------------------------------
constexpr int kMaxRanks = 16;
constexpr int kX1Words = 32;
constexpr int kX2Stride = ((3 * MPPI_MAX_TIME_STEPS + 2 + 15) / 16) * 16;
constexpr int kBoxX1 = 0;                                   // in packets
constexpr int kBoxX2 = kMaxRanks * kX1Words;
constexpr int kBoxPackets = kBoxX2 + kMaxRanks * kX2Stride;
constexpr int kBoxWords = 2 * kBoxPackets;                  // the allocation, in 32-bit words
constexpr long long kSpinLimitCycles = 4000000000LL;        // ~2 s at 1.965 GHz

struct PeerComm
{
  uint2 * box[kMaxRanks];      // box[r] = mailbox of rank r as mapped into this process; box[rank] is local memory
  unsigned * seq;              // local: number of completed exchange rounds; the tag of the current round is *seq + 1
  int rank, nranks;            // nranks <= 1: not sharded over peer memory
};

__device__ __forceinline__ unsigned ld_volatile_u32(const unsigned * p)
{
  unsigned v;
  asm volatile ("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_packet(uint2 * p, unsigned value, unsigned tag)
{
  asm volatile ("st.volatile.global.v2.u32 [%0], {%1, %2};" :: "l"(p), "r"(value), "r"(tag) : "memory");
}
__device__ __forceinline__ uint2 ld_packet(const uint2 * p)
{
  uint2 v;
  asm volatile ("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
// bounded spin on a packet in local memory; returns false (and value 0) on time-out
__device__ __forceinline__ bool poll_packet(const uint2 * p, unsigned tag, unsigned & value)
{
  const long long t0 = clock64();
  for (;;) {
    const uint2 v = ld_packet(p);
    if (v.y == tag) {value = v.x; return true;}
    if (clock64() - t0 > kSpinLimitCycles) {value = 0u; return false;}
  }
}

// Persistent per-optimize state shared between kernels (device memory, 1 record per handle).
struct DevState
{
  unsigned furthest_candidate;          // max over trajectories of argmin over path (this iteration)  [exchange 1]
  unsigned any_ok[kMaxCritics];         // obstacle-type critic q saw a non-colliding trajectory       [exchange 1]
  unsigned furthest;                    // CriticData::furthest_reached_path_point
  int furthest_set;
  int fail_flag;
  unsigned ticket;                      // last-block election of the update kernel
  float global_min;                     // stream layout: min over all costs, published by K3's last block
  unsigned comm_error;                  // a peer-memory exchange timed out (sticky until reset)
};

// Read-only data of a launch is loaded through the non-coherent path (ld.global.nc) -- EXCEPT in the fused kernels, whose
// tiles write the device copy of [record | costmap] themselves (zero-copy upload) before other tiles read it in the same
// launch: ld.global.nc is only defined for data that is read-only for the whole kernel, so there the loads are plain
// (coherent) ones, ordered behind the upload flags by fences (rollout_tile_body).  kNc is a compile-time choice.
template<bool kNc, typename V>
__device__ __forceinline__ V ld_ro(const V * p)
{
  if (kNc) {return __ldg(p);}
  return *p;
}

// ---------------------------------------------------------------------------------------------------
// nav2_costmap_2d::Costmap2D::worldToMap restated; all fp64, inputs are fp32 poses widened.
// Returns the flat cell index my*size_x+mx or -1 (off-map).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int world_to_cell(
  double wx, double wy, double ox, double oy, double res, unsigned size_x, unsigned size_y, unsigned & mx, unsigned & my)
{
  if (wx < ox || wy < oy) {return -1;}
  const double qx = __ddiv_rn(wx - ox, res);
  const double qy = __ddiv_rn(wy - oy, res);
  if (!(qx < static_cast<double>(size_x)) || !(qy < static_cast<double>(size_y))) {return -1;}
  mx = static_cast<unsigned>(qx);
  my = static_cast<unsigned>(qy);
  return static_cast<int>(my * size_x + mx);
}

// worldToMap for a rollout pose, filtered: the cell is first computed in fp32,
//   qf = fl32(fl32(xf - fl32(ox)) * fl32(1/res)),
// whose distance to the reference's fp64 quotient Q = fl64(fl64(double(xf) - ox) / res) is bounded by
//   |qf - Q| <= |Q| * 3.01 * 2^-24 + |ox| / res * 2^-24 * 1.001   (three fp32 roundings + the rounding of ox),
// a bound the host evaluates per cycle as cell_eps_{x,y} (with margin, build_params).  If qf is farther than
// that from every integer, floor(qf) == trunc(Q) and "qf < 0" == "wx < ox", so the fp32 answer IS the
// reference's answer; otherwise (a pose within ~1e-4 cell of a cell edge, or outside the fp32 trick's range)
// the reference's own fp64 arithmetic decides (world_to_cell_slow).  Bit-exact by construction, ~16 fp32
// instructions instead of ~55 fp64/conversion instructions per pose.
struct CellGrid
{
  float oxf, oyf, invf, half_minus_eps_x, half_minus_eps_y;   // 0.5 - error bound in cells (<= 0: always the slow path)
  unsigned size_x, size_y;
};

__device__ __noinline__ int world_to_cell_slow(float xf, float yf, const double * __restrict__ geom, unsigned size_x, unsigned size_y)
{
  // geom = &DevParams::res = {res, ox, oy}
  unsigned mx, my;
  return world_to_cell(static_cast<double>(xf), static_cast<double>(yf), geom[1], geom[2], geom[0], size_x, size_y, mx, my);
}

// floor of q without conversion instructions: adding 1.5 * 2^23 with round-down leaves floor(q) in the low mantissa
// bits (exact for |q| < 2^22; beyond that the decoded integer is >= 2^22 in magnitude, i.e. off any map).
// frac = q - floor(q) is exact.
__device__ __forceinline__ void floor_magic(float q, int & i, float & frac)
{
  const float t = __fadd_rd(q, 12582912.0f);
  i = __float_as_int(t) - 0x4B400000;
  frac = __fsub_rn(q, __fsub_rn(t, 12582912.0f));
}

// The fp32 half of world_to_cell_fast on its own: the candidate cell and whether it is certain.  The stream kernel
// evaluates it for the four poses of a chunk and takes ONE branch to the fp64 path when any of them is uncertain
// (~1e-4 of the poses), instead of one branch per pose.
__device__ __forceinline__ int world_to_cell_try(float xf, float yf, const CellGrid & cg, bool & sure)
{
  const float qx = __fmul_rn(__fsub_rn(xf, cg.oxf), cg.invf);
  const float qy = __fmul_rn(__fsub_rn(yf, cg.oyf), cg.invf);
  int mx, my;
  float fx, fy;
  floor_magic(qx, mx, fx);
  floor_magic(qy, my, fy);
  sure = fabsf(__fsub_rn(fx, 0.5f)) < cg.half_minus_eps_x && fabsf(__fsub_rn(fy, 0.5f)) < cg.half_minus_eps_y;
  if (static_cast<unsigned>(mx) >= cg.size_x || static_cast<unsigned>(my) >= cg.size_y) {return -1;}
  return my * static_cast<int>(cg.size_x) + mx;
}

// The same for callers that send EVERYTHING unusual down one slow branch (the stream kernel's chunk): `plain` is set when
// the fp32 cell is certain AND on the map; the return value is then the flat index and needs no off-map test.  Otherwise
// the value is meaningless and world_to_cell_fast decides.
__device__ __forceinline__ int world_to_cell_plain(float xf, float yf, const CellGrid & cg, bool & plain)
{
  const float qx = __fmul_rn(__fsub_rn(xf, cg.oxf), cg.invf);
  const float qy = __fmul_rn(__fsub_rn(yf, cg.oyf), cg.invf);
  int mx, my;
  float fx, fy;
  floor_magic(qx, mx, fx);
  floor_magic(qy, my, fy);
  plain = fabsf(__fsub_rn(fx, 0.5f)) < cg.half_minus_eps_x && fabsf(__fsub_rn(fy, 0.5f)) < cg.half_minus_eps_y &&
    static_cast<unsigned>(mx) < cg.size_x && static_cast<unsigned>(my) < cg.size_y;
  return my * static_cast<int>(cg.size_x) + mx;
}

__device__ __forceinline__ int world_to_cell_fast(float xf, float yf, const CellGrid & cg, const double * __restrict__ geom)
{
  const float qx = __fmul_rn(__fsub_rn(xf, cg.oxf), cg.invf);
  const float qy = __fmul_rn(__fsub_rn(yf, cg.oyf), cg.invf);
  int mx, my;
  float fx, fy;
  floor_magic(qx, mx, fx);
  floor_magic(qy, my, fy);
  // farther than the error bound from both edges of the cell on both axes?  (NaN and out-of-range fail the test or
  // decode to an off-map index; either way the answer below is the reference's)
  const bool sure = fabsf(__fsub_rn(fx, 0.5f)) < cg.half_minus_eps_x && fabsf(__fsub_rn(fy, 0.5f)) < cg.half_minus_eps_y;
  if (!sure) {return world_to_cell_slow(xf, yf, geom, cg.size_x, cg.size_y);}
  if (static_cast<unsigned>(mx) >= cg.size_x || static_cast<unsigned>(my) >= cg.size_y) {return -1;}
  return my * static_cast<int>(cg.size_x) + mx;
}

// FootprintCollisionChecker::lineCost over nav2_util::LineIterator (integer Bresenham, both ends included).
// The reference walks the cells one by one and returns LETHAL_OBSTACLE at the first lethal cell, otherwise the maximum of
// all cells: the cost of a line is a function of the SET of its cells (lethal if any cell is, else the maximum), so the
// cells are fetched kLineBatch at a time - the loads of a batch are in flight together instead of one L1/L2 round trip
// per cell behind an exit test (the footprint checks of a boxed-in robot were 85 % of the stream rollout's time that
// way) - and the walk stops behind the first batch that holds a lethal cell.  Cells past the end of the line are not
// dereferenced.  The integer stepping is the reference's, cell for cell.
// Measured against it in the boxed-in config 3 (profiles/README.md, K2 per cycle): the slots beyond the end reading the end
// cell again so that every load is unconditional, 153 against 150 us (batches of 6 or 4: 156 us); the cells of a batch in
// closed form, index_k = index_0 + k inc2 + floor((den / 2 + k numadd) / den) inc1 with an exact fp32 floor (no serial index
// chain, but 38.6 M instead of 34.6 M warp instructions): 176 against 153 us under ncu.
constexpr int kLineBatch = 8;
template<bool kNc>
__device__ __forceinline__ int line_cost(const uint8_t * cm, unsigned size_x, int x0, int y0, int x1, int y1)
{
  int deltax = abs(x1 - x0), deltay = abs(y1 - y0);
  int xinc1, xinc2, yinc1, yinc2;
  if (x1 >= x0) {xinc1 = 1; xinc2 = 1;} else {xinc1 = -1; xinc2 = -1;}
  if (y1 >= y0) {yinc1 = 1; yinc2 = 1;} else {yinc1 = -1; yinc2 = -1;}
  int den, num, numadd, numpixels;
  if (deltax >= deltay) {
    xinc1 = 0; yinc2 = 0; den = deltax; num = deltax / 2; numadd = deltay; numpixels = deltax;
  } else {
    xinc2 = 0; yinc1 = 0; den = deltay; num = deltay / 2; numadd = deltax; numpixels = deltay;
  }
  // flat index of the cell and its two increments (the minor step is taken when the error term overflows)
  const int sx = static_cast<int>(size_x);
  int idx = y0 * sx + x0;
  const int inc1 = yinc1 * sx + xinc1, inc2 = yinc2 * sx + xinc2;
  int cost = 0;
  for (int cur = 0; cur <= numpixels; cur += kLineBatch) {
    int c[kLineBatch];
#pragma unroll
    for (int k = 0; k < kLineBatch; ++k) {
      c[k] = cur + k <= numpixels ? static_cast<int>(ld_ro<kNc>(cm + static_cast<unsigned>(idx))) : 0;
      num += numadd;
      if (num >= den) {num -= den; idx += inc1;}
      idx += inc2;
    }
    bool lethal = false;
#pragma unroll
    for (int k = 0; k < kLineBatch; ++k) {lethal = lethal || c[k] == LETHAL_OBSTACLE; cost = max(cost, c[k]);}
    if (lethal) {return LETHAL_OBSTACLE;}
  }
  return cost;
}

// FootprintCollisionChecker::footprintCostAtPose + footprintCost.  P is the record in GLOBAL memory (the polygon
// is not part of the hot copy); the scalars come from the caller's registers.  kNc: see ld_ro.
// The reference interleaves "map the next vertex, return LETHAL_OBSTACLE if it is off the map" with the line walks; every
// exit it takes for an off-map vertex returns the same value whatever the lines before it held, so the vertices are mapped
// first, in a loop without exits: the two fp64 divisions per vertex (worldToMap) of all vertices overlap instead of each
// waiting behind the previous line's loads.  Then the lines in the reference's order (0-1, 1-2, ..., and the closing line
// from vertex 0 to the last one, in THAT direction: Bresenham is not symmetric), with its running maximum and its exit.
template<bool kNc>
__device__ __noinline__ int footprint_cost_at_pose(
  const DevParams * P, int n, double ox, double oy, double res, unsigned size_x, unsigned size_y,
  const uint8_t * cm, float xf, float yf, float thf)
{
  const double x = xf, y = yf, th = thf;
  double sin_th, cos_th;
  sincos(th, &sin_th, &cos_th);
  int vx[MPPI_MAX_FOOTPRINT], vy[MPPI_MAX_FOOTPRINT];
  bool off = false;
  n = max(n, 1);   // an empty polygon reads vertex 0 of the record like the reference reads footprint[0]
#pragma unroll 4
  for (int i = 0; i < n; ++i) {
    const double fx = ld_ro<kNc>(&P->fp_x[i]), fy = ld_ro<kNc>(&P->fp_y[i]);
    const double wx = x + (__dmul_rn(fx, cos_th) - __dmul_rn(fy, sin_th));
    const double wy = y + (__dmul_rn(fx, sin_th) + __dmul_rn(fy, cos_th));
    unsigned mx = 0u, my = 0u;
    off = (world_to_cell(wx, wy, ox, oy, res, size_x, size_y, mx, my) < 0) || off;
    vx[i] = static_cast<int>(mx); vy[i] = static_cast<int>(my);
  }
  if (off) {return LETHAL_OBSTACLE;}
  int footprint_cost = 0;
  for (int i = 0; i + 1 < n; ++i) {
    footprint_cost = max(line_cost<kNc>(cm, size_x, vx[i], vy[i], vx[i + 1], vy[i + 1]), footprint_cost);
    if (footprint_cost == LETHAL_OBSTACLE) {return footprint_cost;}
  }
  return max(line_cost<kNc>(cm, size_x, vx[0], vy[0], vx[n - 1], vy[n - 1]), footprint_cost);
}

// CostCritic::inCollision / ObstaclesCritic::inCollision on a byte cost
__device__ __forceinline__ bool in_collision(int cost, bool consider_footprint, bool track_unknown)
{
  if (cost == LETHAL_OBSTACLE) {return true;}
  if (cost == INSCRIBED_INFLATED_OBSTACLE) {return !consider_footprint;}
  if (cost == NO_INFORMATION) {return !track_unknown;}
  return false;
}

// utils::normalize_angles on one element: fmod(a + pi, 2 pi) in double, <= 0 -> + pi else - pi
__device__ __forceinline__ double normalize_angle_d(double a)
{
  const double two_pi = 6.283185307179586476925286766559;
  const double pi = 3.14159265358979323846;
  double v = a + pi;
  double theta;
  if (v >= 0.0 && v < two_pi) {
    theta = v;
  } else if (v >= two_pi && v < 2.0 * two_pi) {
    theta = v - two_pi;          // exact (Sterbenz), equals fmod
  } else if (v < 0.0 && v > -two_pi) {
    theta = v;                   // fmod keeps the sign of the dividend
  } else {
    theta = fmod(v, two_pi);
  }
  return theta <= 0.0 ? theta + pi : theta - pi;
}

// costs += pow(value, power) as the reference's xtensor expression evaluates it (pow and the sum in double)
__device__ __forceinline__ float add_pow(float total, float value, unsigned power)
{
  if (power == 1u) {return __fadd_rn(total, value);}
  return static_cast<float>(static_cast<double>(total) + pow(static_cast<double>(value), static_cast<double>(power)));
}

// the same, with the power != 1 branch out of line: for code that runs once per launch (tile / fused kernels), where the
// inlined double-precision pow only makes the instruction footprint larger (these kernels stall on instruction fetch)
__device__ __noinline__ float add_pow_slow(float total, float value, unsigned power)
{
  return static_cast<float>(static_cast<double>(total) + pow(static_cast<double>(value), static_cast<double>(power)));
}
__device__ __forceinline__ float add_pow_c(float total, float value, unsigned power)
{
  if (power == 1u) {return __fadd_rn(total, value);}
  return add_pow_slow(total, value, power);
}

// sqrt for cost terms (1e-4 tolerance): one MUFU instead of the IEEE sequence
__device__ __forceinline__ float sqrt_approx(float v)
{
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

__device__ __forceinline__ float warp_min(float v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));}
  return v;
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {v += __shfl_xor_sync(0xffffffffu, v, o);}
  return v;
}
__device__ __forceinline__ unsigned warp_max_u(unsigned v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {v = max(v, __shfl_xor_sync(0xffffffffu, v, o));}
  return v;
}

}  // namespace mppi
