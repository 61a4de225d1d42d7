// mppi_api.cu -- the C ABI of include/mppi_b200.h over the sm_100a kernels of mppi_kernels.cuh.
//
// Host responsibilities (all O(N) or O(critics) scalar work per cycle, never O(B)):
//   * keep the Optimizer state the reference keeps between cycles (control sequence, constraints, noise)
//   * evaluate the per-cycle scalar gates of the critics exactly as the reference does on the host
//     (withinPositionGoalTolerance, posePointAngle, findCircumscribedCost, ...), pack them with the path
//     into one pinned record, and ship record + costmap with two async copies
//   * launch K2 -> [exchange 1] -> K3 -> [exchange 2 -> K4], read back the 3T+2 floats of the result
// There is no CPU implementation of the hot path in this file: without a CUDA device every call fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <time.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "mppi_kernels.cuh"

using namespace mppi;

namespace
{

struct NcclApi
{
  void * lib{nullptr};
  ncclResult_t (*GetUniqueId)(ncclUniqueId *){nullptr};
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int){nullptr};
  ncclResult_t (*CommDestroy)(ncclComm_t){nullptr};
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t){nullptr};
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t){nullptr};
  const char * (*GetErrorString)(ncclResult_t){nullptr};
  bool load(std::string & err)
  {
    if (lib) {return true;}
    // by soname: if torch (or anything else) already mapped an NCCL in this process, that copy is reused
    lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) {err = std::string("dlopen libnccl.so.2: ") + dlerror(); return false;}
    GetUniqueId = reinterpret_cast<decltype(GetUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
    CommInitRank = reinterpret_cast<decltype(CommInitRank)>(dlsym(lib, "ncclCommInitRank"));
    CommDestroy = reinterpret_cast<decltype(CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
    AllReduce = reinterpret_cast<decltype(AllReduce)>(dlsym(lib, "ncclAllReduce"));
    AllGather = reinterpret_cast<decltype(AllGather)>(dlsym(lib, "ncclAllGather"));
    GetErrorString = reinterpret_cast<decltype(GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
    if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllReduce || !AllGather) {
      err = "libnccl.so.2 lacks a required symbol";
      return false;
    }
    return true;
  }
};
NcclApi g_nccl;

struct Constraints {float vx_max, vx_min, vy, wz;};

}  // namespace

struct mppi_handle
{
  mppi_config cfg;
  Constraints base, cur;
  std::vector<mppi_critic_desc> critics;
  std::vector<uint8_t> scratch_gate;       // build_params scratch (no allocation in the steady state)
  std::vector<uint16_t> scratch_prefix;
  std::vector<int> scratch_next;
  mppi_robot_desc robot;
  int B{0}, T{0};
  int device{0};
  cudaStream_t stream{nullptr};
  cudaEvent_t ev0{nullptr}, ev1{nullptr};
  cudaEvent_t pev[4]{nullptr, nullptr, nullptr, nullptr};   // profiling: before K2, after K2, after K3, after exchange 2
  bool profiling{false};
  bool timing{true};           // bracket every cycle with two events and report device_ms (mppi_set_timing)
  float prof_ms[4]{0.f, 0.f, 0.f, 0.f};
  uint64_t launches{0};
  uint64_t h2d_bytes{0}, d2h_bytes{0};
  // device
  float * d_noise[3]{nullptr, nullptr, nullptr};
  // one upload buffer per side, [cycle record (kParamsCapacity reserved) | costmap]: the record is copied alone
  // (resident costmap) or record + costmap in ONE async copy: the costmap is staged right behind the bytes of the record
  // that are copied (d_costmap = d_params + params_copy_bytes rounded up to 256)
  uint8_t * d_costmap{nullptr};
  size_t costmap_capacity{0};
  char * d_params{nullptr};
  float * d_cs{nullptr};
  float * d_crit_rows{nullptr};
  float * d_samples[3]{nullptr, nullptr, nullptr};
  float * d_end_xy{nullptr};
  float * d_spill[3]{nullptr, nullptr, nullptr};
  int * d_cells{nullptr};
  float * d_costs{nullptr};
  float * d_partials{nullptr};
  unsigned * d_ws_done{nullptr};         // per row group of the weighted-sums kernel: blocks finished (last one merges)
  CUtensorMap noise_map[3];           // TMA descriptors of the time-major noise planes (stream layout, weighted_sums_tma_kernel)
  bool pdl_enabled{true};             // MPPI_PDL=0: ordinary (fully serialised) launches of the stream layout's post-rollout kernels
  int scan_mode{0};                   // MPPI_SCAN=warp: experiment, warp-shuffle prefix scans in the tile kernels (not the parity path)
  bool ws_tma_enabled{true};             // MPPI_WS_TMA=0: the register-staged weighted-sums kernel (always used when B % 4 != 0)
  bool ws_tma_ok{false};                 // the TMA-fed weighted-sums kernel can run (B % 4 == 0, descriptors made)
  float * d_rank_partial{nullptr};
  float * d_gathered{nullptr};
  size_t gathered_capacity{0};   // records d_gathered holds (exchange 2: one (3T + 2)-float record per rank / shard)
  float * d_out{nullptr};
  DevState * d_st{nullptr};
  float * d_inj[6]{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // score / integrate scratch, lazy
  float * d_tmp{nullptr};                                                   // [B][T] transposition scratch, lazy
  // pinned host
  char * h_params{nullptr};
  uint8_t * h_costmap{nullptr};
  size_t h_costmap_capacity{0};
  float * h_out{nullptr};
  // state
  size_t params_bytes{0};
  uint64_t noise_stream{0};
  uint32_t want_mask{0};
  bool cycle_uploaded{false};
  bool spilled_traj{false}, spilled_cells{false}, have_rows{false};
  DevParams last;   // host copy of the last uploaded record
  int segments_override{0};
  int stream_threads_override{0};
  // fused small-batch kernel: packet buffers of the in-GPU exchanges, launch epoch (device + host mirror), result packets
  uint2 * d_pk{nullptr};                  // [G] exchange-1 packets, then [G][3T + 2] record packets
  unsigned * d_fepoch{nullptr};           // completed fused launches (never reset: tags do not repeat)
  uint32_t fepoch_host{0};                // host mirror of *d_fepoch once everything enqueued has run
  uint2 * h_res{nullptr};                 // pinned + mapped: [3T + 8] result packets written by the kernels
  bool zero_copy_now{false};              // this cycle's fused kernel pulls the upload out of pinned host memory itself
  bool wait_packets{false};               // the cycle in flight delivers its result as packets (no D2H copy, no stream sync)
  // multi-robot batch (mppi_batch_bind): the bound handles share the leader's stream, so that ONE launch can serve all
  // of them (tile_fused_batch_kernel) and every later operation on any of them is still ordered behind it
  mppi_handle * batch_leader{nullptr};    // non-null for every bound handle (the leader points to itself)
  cudaStream_t own_stream{nullptr};       // a follower's own stream while it borrows the leader's
  mppi_handle * ev_src{nullptr};          // whose ev0 / ev1 bracket the cycle in flight (the leader's after a batched launch)
  std::vector<mppi_handle *> batch_group; // leader only, in bind order
  cudaStream_t copy_stream{nullptr};      // leader only (stream-layout group): the chunk uploads ride here, beside the previous chunk's kernels
  cudaEvent_t ev_upload[8]{};             // leader only: upload of chunk c done (c modulo 8)
  FusedJob * h_jobs{nullptr};             // leader only: job table, pinned ...
  FusedJob * d_jobs{nullptr};             // ... and its device copy (re-sent only when an entry changes)
  std::vector<char> jobs_sent;            // what the device copy holds
  unsigned * d_ticket{nullptr};           // leader only: ticket counter of the batch kernel (never reset)
  uint32_t ticket_base{0};                // tickets drawn by all earlier batched launches
  int batch_mode{0};                      // leader: 1 = tile layout, ticketed fused kernel; 2 = stream layout, four batched kernels
  char * arena_h{nullptr};                // leader, mode 2: the [record | costmap] buffers of all members, one slice each,
  char * arena_d{nullptr};                //   so that the whole group uploads with ONE strided copy
  size_t arena_slice{0};
  bool params_in_arena{false};            // member: h_params / d_params point into the leader's arena
  uint32_t batch_tag{0};                  // leader, mode 2: counter behind the tag of the group's result packets
  uint32_t result_tag{0};                 // tag the cycle in flight delivers its result packets with
  // caller memory registered as pinned (mppi_register_costmap_memory): a costmap inside such a range is copied to the
  // device straight from the caller's buffer, without the staging memcpy
  std::vector<std::pair<const char *, size_t>> pinned_ranges;
  const uint8_t * costmap_direct{nullptr};   // this cycle's costmap source when it is copied directly
  uint64_t host_ns[8]{0, 0, 0, 0, 0, 0, 0, 0};   // host-side time of the steady-state call by phase (mppi_debug_get_host_ns)
  bool zero_copy_enabled{true};   // MPPI_ZERO_COPY=0 disables
  bool coop_launch{true};
  bool packets_enabled{true};     // MPPI_STREAM_PACKETS=0: the stream layout copies its result back and synchronises
  bool fused_enabled{true};    // small batches: one cooperative launch per iteration (tile_fused_kernel); MPPI_FUSED=0 disables
  int fused_key_N{-1};         // path size the cached decision below was taken for (the shared-memory size depends on it)
  bool fused_fits{false};      // the whole grid is co-resident (a cooperative launch needs that)
  int num_sms{0};
  bool stream_layout{false};   // large batches: time-major noise + thread-per-trajectory K2 + GEMV-style weighted sums
  int upd_blocks{0};
  // CUDA graphs of the steady-state cycle: [0] kernels + D2H (resident inputs), [1] H2D + kernels + D2H
  // captured graphs: slot = (with_upload ? 1 : 0) + 2 * tail_mode
  // (+ 6 when the cycle is timed: the two event records are nodes of the graph, so that device_ms does not contain the
  //  host's gap between recording an event and launching the graph)
  cudaGraphExec_t gexec[12]{};
  size_t gkey_params[12]{}, gkey_costmap[12]{};
  unsigned gkey_inst[12]{};
  int gkey_fused[12]{};   // fused kernel: shared-memory key (path capacity, PathAlign samples); -1 = two-kernel path
  int tail_mode{0};            // 0: optimize only, 1: + evalControl tail, 2: + tail with shiftControlSequence
  // peer-memory exchange (one process per GPU; mppi_comm_get_mailbox_handle / mppi_comm_connect_peers)
  uint2 * d_mailbox{nullptr};             // this rank's mailbox (kBoxPackets packets)
  unsigned * d_seq{nullptr};              // completed exchange rounds (survives mppi_reset: tags never repeat)
  uint2 * peer_box[kMaxRanks]{};          // mailboxes of all ranks as mapped here; [rank] == d_mailbox
  bool peer_mode{false};
  int vis_b_step{0}, vis_t_step{0};       // mppi_set_visualization
  float * d_vis{nullptr};
  size_t vis_capacity{0};
  bool vis_valid{false};
  float * d_hist{nullptr};     // control_history_ [4][3] (vx, vy, wz), optimizer.hpp:251
  unsigned long long * d_epoch{nullptr};   // regenerate_noises: Philox stream index of the next draw (device copy of noise_stream)
  cudaEvent_t ev_result{nullptr};          // regenerate_noises: result is in host memory (the redraw may still be running)
  bool capturing{false};
  bool use_graph{true};
  size_t costmap_bytes{0}, params_copy_bytes{0};
  // sharding
  ncclComm_t comm{nullptr};
  int rank{0}, nranks{1};
  std::string err;
};

namespace
{

// record + per path point: x, y, yaw, D (floats), PathAngle gate byte, validity byte, invalid-prefix uint16 (+ slack)
constexpr size_t kParamsCapacity = sizeof(DevParams) + MPPI_MAX_PATH_POINTS * (4 * sizeof(float) + 4) + 256;

#define CUDA_TRY(h, expr)                                                                          \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      (h)->err = std::string(#expr) + ": " + cudaGetErrorString(e_);                               \
      return MPPI_E_CUDA;                                                                          \
    }                                                                                              \
  } while (0)

#define NCCL_TRY(h, expr)                                                                          \
  do {                                                                                             \
    ncclResult_t r_ = (expr);                                                                      \
    if (r_ != ncclSuccess) {                                                                       \
      (h)->err = std::string(#expr) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error"); \
      return MPPI_E_NCCL;                                                                          \
    }                                                                                              \
  } while (0)

inline uint64_t now_ns()
{
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return static_cast<uint64_t>(ts.tv_sec) * 1000000000ull + static_cast<uint64_t>(ts.tv_nsec);
}

mppi_status fail(mppi_handle * h, mppi_status s, const std::string & msg)
{
  if (h) {h->err = msg;}
  return s;
}

bool holonomic(const mppi_handle * h) {return h->cfg.motion_model == MPPI_MODEL_OMNI;}

// ---- host-side scalar helpers, restating the reference's host code --------------------------------
// utils::withinPositionGoalTolerance(float, ...) utils.hpp:233-249
bool within_tolerance(float pose_tolerance, double rx, double ry, double gx, double gy)
{
  const double dist_sq = std::pow(gx - rx, 2) + std::pow(gy - ry, 2);
  const float pose_tolerance_sq = pose_tolerance * pose_tolerance;
  return dist_sq < pose_tolerance_sq;
}
// utils::withinPositionGoalTolerance(GoalChecker*, ...) utils.hpp:201-224
bool within_checker_tolerance(double tol, double rx, double ry, double gx, double gy)
{
  if (tol >= 0.0) {
    const double dx = rx - gx, dy = ry - gy;
    if (dx * dx + dy * dy < tol * tol) {return true;}
  }
  return false;
}
double normalize_angle(double angle)
{
  const double result = std::fmod(angle + M_PI, 2.0 * M_PI);
  if (result <= 0.0) {return result + M_PI;}
  return result - M_PI;
}
// utils::posePointAngle utils.hpp:417-434
float pose_point_angle(double pose_xd, double pose_yd, double pose_yawd, double point_x, double point_y, bool forward_preference)
{
  const float pose_x = pose_xd, pose_y = pose_yd, pose_yaw = pose_yawd;
  const float yaw = atan2f(point_y - pose_y, point_x - pose_x);
  if (!forward_preference) {
    return std::min(
      fabs(normalize_angle(static_cast<double>(pose_yaw) - yaw)),
      fabs(normalize_angle(normalize_angle(pose_yaw + M_PI) - yaw)));
  }
  return fabs(normalize_angle(static_cast<double>(pose_yaw) - yaw));
}
// InflationLayer::computeCost + {Obstacles,Cost}Critic::findCircumscribedCost
float circumscribed_cost(const mppi_robot_desc & robot, double resolution)
{
  double result = -1.0;
  if (robot.inflation_layer_found) {
    const double distance = robot.circumscribed_radius / resolution;
    unsigned char cost = 0;
    if (distance == 0) {
      cost = LETHAL_OBSTACLE;
    } else if (distance * resolution <= robot.inscribed_radius) {
      cost = INSCRIBED_INFLATED_OBSTACLE;
    } else {
      const double factor = std::exp(-1.0 * robot.inflation_cost_scaling_factor * (distance * resolution - robot.inscribed_radius));
      cost = static_cast<unsigned char>((INSCRIBED_INFLATED_OBSTACLE - 1) * factor);
    }
    result = cost;
  }
  return static_cast<float>(result);
}

const mppi_critic_desc * find_kind(const mppi_handle * h, int kind, int * idx)
{
  for (size_t i = 0; i < h->critics.size(); ++i) {
    if (h->critics[i].kind == kind) {*idx = static_cast<int>(i); return &h->critics[i];}
  }
  *idx = -1;
  return nullptr;
}

void set_common(CriticCommon & c, const mppi_critic_desc * d, int idx, bool gate)
{
  c.idx = idx;
  c.on = (d && d->enabled && gate) ? 1 : 0;
  c.power = d ? d->cost_power : 1u;
  c.weight = d ? d->cost_weight : 0.0f;
}

// Fill the per-cycle record.  `in` may be null for integrate-only calls (mode 1).
mppi_status build_params(mppi_handle * h, const mppi_cycle_in * in, int mode, unsigned preset_furthest, bool critics_active,
  const float * first_pose = nullptr)
{
  DevParams & p = *reinterpret_cast<DevParams *>(h->h_params);
  std::memset(&p, 0, sizeof(p));
  const mppi_config & cfg = h->cfg;
  p.B = h->B; p.T = h->T;
  p.holonomic = holonomic(h) ? 1 : 0;
  p.model = cfg.motion_model;
  p.mode = mode;
  p.dt = cfg.model_dt;
  p.min_turning_r = cfg.ackermann_min_turning_r;
  p.temperature = cfg.temperature;
  p.gamma_vx = cfg.gamma / powf(cfg.vx_std, 2);
  p.gamma_vy = cfg.gamma / powf(cfg.vy_std, 2);
  p.gamma_wz = cfg.gamma / powf(cfg.wz_std, 2);
  p.c_vx_max = h->cur.vx_max; p.c_vx_min = h->cur.vx_min; p.c_vy = h->cur.vy; p.c_wz = h->cur.wz;
  p.preset_furthest = preset_furthest;
  p.track_unknown = h->robot.track_unknown;
  p.want_cells = (h->want_mask & MPPI_WANT_CELLS) ? 1 : 0;
  p.want_critic_rows = (h->want_mask & MPPI_WANT_CRITIC_COSTS) ? 1 : 0;
  p.vis_b_step = h->vis_b_step; p.vis_t_step = h->vis_t_step;
  p.vis_nb = h->vis_b_step > 0 ? (h->B + h->vis_b_step - 1) / h->vis_b_step : 0;
  p.fp_n = h->robot.footprint_size;
  for (int i = 0; i < p.fp_n; ++i) {p.fp_x[i] = h->robot.footprint_x[i]; p.fp_y[i] = h->robot.footprint_y[i];}

  const double rx = in->pose_x, ry = in->pose_y, gx = in->goal_x, gy = in->goal_y;
  p.pose_x = rx; p.pose_y = ry;
  p.yaw0 = static_cast<float>(in->pose_yaw);                  // const float initial_yaw = tf2::getYaw(...)
  mppi_det_sincosf(p.yaw0, &p.sin0, &p.cos0);
  p.speed_vx = static_cast<float>(in->speed_vx); p.speed_vy = static_cast<float>(in->speed_vy);
  p.speed_wz = static_cast<float>(in->speed_wz);
  p.goal_x = gx; p.goal_y = gy;
  const int N = in->path_size;
  if (N < 1 || N > MPPI_MAX_PATH_POINTS) {return fail(h, MPPI_E_CONFIG, "path_size must be in [1, MPPI_MAX_PATH_POINTS]");}
  if (!in->path_x || !in->path_y || !in->path_yaw) {return fail(h, MPPI_E_CONFIG, "null path arrays");}
  p.N = N;
  p.goal_yaw = in->path_yaw[N - 1];
  p.size_x = in->costmap.size_x; p.size_y = in->costmap.size_y;
  if (p.size_x >= (1u << 22) || p.size_y >= (1u << 22)) {return fail(h, MPPI_E_CONFIG, "costmap side must be < 2^22 cells");}
  p.res = in->costmap.resolution; p.ox = in->costmap.origin_x; p.oy = in->costmap.origin_y;
  // fp32 filter of worldToMap (mppi_device.cuh world_to_cell_fast): operands and rigorous error bounds in cells
  p.cell_oxf = static_cast<float>(p.ox);
  p.cell_oyf = static_cast<float>(p.oy);
  p.cell_invf = static_cast<float>(1.0 / p.res);
  {
    const double u = 5.9604644775390625e-08;   // 2^-24
    p.cell_eps_x = static_cast<float>(((static_cast<double>(p.size_x) + 2.0) * 3.5 + std::fabs(p.ox) / p.res * 1.1) * u + 1.0e-6);
    p.cell_eps_y = static_cast<float>(((static_cast<double>(p.size_y) + 2.0) * 3.5 + std::fabs(p.oy) / p.res * 1.1) * u + 1.0e-6);
  }

  // path arrays behind the struct: x, y, yaw, arc-length prefix D (path_align_critic.cpp:83-90), PathAngle gate bytes
  float * tail = reinterpret_cast<float *>(h->h_params + sizeof(DevParams));
  p.off_path_x = 0; p.off_path_y = N; p.off_path_yaw = 2 * N; p.off_path_D = 3 * N;
  std::memcpy(tail, in->path_x, sizeof(float) * N);
  std::memcpy(tail + N, in->path_y, sizeof(float) * N);
  std::memcpy(tail + 2 * N, in->path_yaw, sizeof(float) * N);
  float * D = tail + 3 * N;
  D[0] = 0.0f;
  for (int i = 1; i < N; ++i) {
    const float dx = in->path_x[i] - in->path_x[i - 1];
    const float dy = in->path_y[i] - in->path_y[i - 1];
    const float curr_dist = sqrtf(dx * dx + dy * dy);
    D[i] = D[i - 1] + curr_dist;
  }
  // host-made tables behind the path arrays: valid[n16] | flags[n16] | follow_idx[N] (uint16); see DevParams
  const int n16 = ((N + 15) / 16) * 16;
  uint8_t * valid = reinterpret_cast<uint8_t *>(tail + 4 * N);
  uint8_t * flags = valid + n16;
  uint16_t * follow_tab = reinterpret_cast<uint16_t *>(valid + 2 * n16);
  std::memset(valid, 0, 2 * n16 + sizeof(uint16_t) * N);
  std::vector<uint8_t> & gate = h->scratch_gate;              // PathAngle gate per candidate target index
  std::vector<uint16_t> & invalid_before = h->scratch_prefix; // number of invalid points among [0, j)
  gate.assign(N, 0);
  invalid_before.assign(N + 1, 0);
  h->params_bytes = sizeof(DevParams) + sizeof(float) * 4 * N + 2 * n16 + sizeof(uint16_t) * N;
  // copy size rounded up to 64 path points so that the captured graph survives small changes of the pruned path
  {
    const size_t n64 = std::min<size_t>(MPPI_MAX_PATH_POINTS, ((static_cast<size_t>(N) + 63) / 64) * 64);
    h->params_copy_bytes = std::min(kParamsCapacity, sizeof(DevParams) + 20 * n64 + 128);
    h->params_copy_bytes = std::max(h->params_copy_bytes, (h->params_bytes + 15) & ~static_cast<size_t>(15));
  }
  // utils::findPathCosts (utils.hpp:361-394): validity of every path point but the last, against the costmap the
  // caller holds for this cycle; prefix counts of the invalid ones for PathAlign's occupancy gate
  for (int j = 0; j < N; ++j) {
    bool ok = false;
    if (j < N - 1 && in->costmap.cells) {
      const double wx = in->path_x[j], wy = in->path_y[j];
      if (!(wx < p.ox || wy < p.oy)) {
        const double qx = (wx - p.ox) / p.res, qy = (wy - p.oy) / p.res;
        if (qx < static_cast<double>(p.size_x) && qy < static_cast<double>(p.size_y)) {
          const unsigned mx = static_cast<unsigned>(qx), my = static_cast<unsigned>(qy);
          if (mx < p.size_x && my < p.size_y) {
            const int c = in->costmap.cells[static_cast<size_t>(my) * p.size_x + mx];
            ok = !(c == LETHAL_OBSTACLE || c == INSCRIBED_INFLATED_OBSTACLE || (c == NO_INFORMATION && !h->robot.track_unknown));
          }
        }
      }
    }
    valid[j] = ok ? 1 : 0;
    invalid_before[j + 1] = static_cast<uint16_t>(invalid_before[j] + (ok ? 0 : 1));
  }
  // utils::findPathTrajectoryInitialPoint (utils.hpp:327-344): closest path point to trajectory 0's first pose.  In the
  // rollout modes that pose is the same for every trajectory (state velocities of step 0 are the robot speed), so the
  // host evaluates it with the kernels' own arithmetic (this TU's host pass is built with -ffp-contract=off).
  {
    float x00, y00;
    if (first_pose) {
      x00 = first_pose[0]; y00 = first_pose[1];
    } else {
      const float dt = cfg.model_dt;
      const float vx0 = p.speed_vx, vy0 = holonomic(h) ? p.speed_vy : 0.0f;
      float dx = vx0 * p.cos0, dy = vx0 * p.sin0;
      if (holonomic(h)) {
        const float a = vy0 * p.sin0, b2 = vy0 * p.cos0;
        dx = dx - a; dy = dy + b2;
      }
      const float tx = dx * dt, ty = dy * dt;
      x00 = static_cast<float>(rx + static_cast<double>(tx));
      y00 = static_cast<float>(ry + static_cast<double>(ty));
    }
    float best = 3.402823466e+38f;
    int best_j = 0;
    for (int j = 0; j < N; ++j) {
      const float dx = in->path_x[j] - x00, dy = in->path_y[j] - y00;
      const float dxx = dx * dx, dyy = dy * dy;
      const float d = dxx + dyy;
      if (d < best) {best = d; best_j = j;}
    }
    p.closest_path_pt = best_j;
    // longest segment and mean spacing of the path (double, from the fp32 coordinates the kernels read)
    double hmax = 0.0, len = 0.0;
    for (int j = 0; j + 1 < N; ++j) {
      const double sx = static_cast<double>(in->path_x[j + 1]) - static_cast<double>(in->path_x[j]);
      const double sy = static_cast<double>(in->path_y[j + 1]) - static_cast<double>(in->path_y[j]);
      const double seg = std::sqrt(sx * sx + sy * sy);
      hmax = std::max(hmax, seg); len += seg;
    }
    p.path_hmax_inv = (hmax > 0.0 && std::isfinite(hmax)) ? static_cast<float>(1.0 / (hmax * 1.00001)) : 0.0f;
    p.path_hmean_inv = (len > 0.0 && std::isfinite(len)) ? static_cast<float>(static_cast<double>(N - 1) / len) : 0.0f;
  }

  p.n_critics = critics_active ? static_cast<int>(h->critics.size()) : 0;
  for (int i = 0; i < kMaxCritics; ++i) {p.kind_of[i] = i < p.n_critics ? h->critics[i].kind : -1;}
  for (CriticCommon * c : {&p.constraint, &p.cost, &p.goal, &p.goal_angle, &p.obst, &p.align, &p.legacy, &p.angle, &p.follow,
      &p.forward, &p.twirl, &p.deadband})
  {
    c->idx = -1; c->on = 0; c->power = 1; c->weight = 0.0f;
  }
  bool any_gate_open = false;
  if (critics_active) {
    int idx;
    const mppi_critic_desc * d;
    if ((d = find_kind(h, MPPI_CRITIC_CONSTRAINT, &idx))) {
      set_common(p.constraint, d, idx, true);
      // constraint_critic.cpp:31-38 : parent parameters at init, not the speed-limited constraints
      const float vx_max = cfg.vx_max, vy_max = cfg.vy_max, vx_min = cfg.vx_min;
      const float min_sgn = vx_min > 0.0 ? 1.0 : -1.0;
      p.max_vel = sqrtf(vx_max * vx_max + vy_max * vy_max);
      p.min_vel = min_sgn * sqrtf(vx_min * vx_min + vy_max * vy_max);
    }
    if ((d = find_kind(h, MPPI_CRITIC_COST, &idx))) {
      set_common(p.cost, d, idx, true);
      p.cost.weight = d->cost_weight / 254.0f;                 // cost_critic.cpp:34
      p.cost_fp = d->consider_footprint; p.cost_critical = d->critical_cost; p.cost_collision = d->collision_cost;
      p.cost_near_goal = within_tolerance(d->near_goal_distance, rx, ry, gx, gy) ? 1 : 0;
      p.cost_possibly_inscribed = circumscribed_cost(h->robot, p.res);
      if (d->enabled && d->consider_footprint && p.fp_n < 1) {return fail(h, MPPI_E_CONFIG, "CostCritic.consider_footprint needs mppi_set_robot");}
    }
    if ((d = find_kind(h, MPPI_CRITIC_GOAL, &idx))) {
      set_common(p.goal, d, idx, within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
    }
    if ((d = find_kind(h, MPPI_CRITIC_GOAL_ANGLE, &idx))) {
      set_common(p.goal_angle, d, idx, within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
    }
    if ((d = find_kind(h, MPPI_CRITIC_OBSTACLES, &idx))) {
      set_common(p.obst, d, idx, true);
      p.obst_fp = d->consider_footprint; p.obst_collision = d->collision_cost;
      p.obst_critical_w = d->critical_weight; p.obst_repulsion_w = d->repulsion_weight;
      p.obst_near_goal = within_tolerance(d->near_goal_distance, rx, ry, gx, gy) ? 1 : 0;
      p.obst_possibly_inscribed = circumscribed_cost(h->robot, p.res);
      if (d->enabled && d->consider_footprint && p.fp_n < 1) {return fail(h, MPPI_E_CONFIG, "ObstaclesCritic.consider_footprint needs mppi_set_robot");}
      // obstacles_critic.cpp:78-80: scale / radius are read only when an inflation layer exists
      const float scale = h->robot.inflation_layer_found ? d->cost_scaling_factor : 0.0f;
      const float infl_r = h->robot.inflation_layer_found ? d->inflation_radius : 0.0f;
      p.obst_repulsion_enabled = !(infl_r == 0.0f || scale == 0.0f);
      if (p.obst_repulsion_enabled) {
        // distanceToObstacle (obstacles_critic.cpp:99-112) tabulated per byte cost; same libm as the oracle
        const float min_radius = h->robot.inscribed_radius;
        for (int fp = 0; fp < 2; ++fp) {
          for (int v = 1; v < 256; ++v) {
            float dist_to_obj = (scale * min_radius - logf(static_cast<float>(v)) + logf(253.0f)) / scale;
            if (!fp) {dist_to_obj -= min_radius;}
            if (dist_to_obj < d->collision_margin_distance) {
              p.obst_lut_crit[fp][v] = d->collision_margin_distance - dist_to_obj;
              p.obst_lut_rep[fp][v] = 0.0f;
            } else {
              p.obst_lut_crit[fp][v] = 0.0f;
              p.obst_lut_rep[fp][v] = infl_r - dist_to_obj;
            }
          }
        }
      }
    }
    if ((d = find_kind(h, MPPI_CRITIC_PREFER_FORWARD, &idx))) {
      set_common(p.forward, d, idx, !within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
    }
    if ((d = find_kind(h, MPPI_CRITIC_TWIRLING, &idx))) {
      set_common(p.twirl, d, idx, !within_checker_tolerance(in->goal_checker_xy_tolerance, rx, ry, gx, gy));
    }
    if ((d = find_kind(h, MPPI_CRITIC_VELOCITY_DEADBAND, &idx))) {
      set_common(p.deadband, d, idx, true);
      p.db_vx = d->deadband_velocities[0]; p.db_vy = d->deadband_velocities[1]; p.db_wz = d->deadband_velocities[2];
    }
    if ((d = find_kind(h, MPPI_CRITIC_PATH_FOLLOW, &idx))) {
      set_common(p.follow, d, idx, N >= 2 && !within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
      p.follow_offset = d->offset_from_furthest;
    }
    if ((d = find_kind(h, MPPI_CRITIC_PATH_ALIGN, &idx))) {
      set_common(p.align, d, idx, !within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
      p.align_offset = d->offset_from_furthest; p.align_step = d->trajectory_point_step;
      p.align_use_yaw = d->use_path_orientations; p.align_max_ratio = d->max_path_occupancy_ratio;
      if (d->enabled && d->trajectory_point_step < 1) {return fail(h, MPPI_E_CONFIG, "PathAlignCritic.trajectory_point_step < 1");}
    }
    if ((d = find_kind(h, MPPI_CRITIC_PATH_ALIGN_LEGACY, &idx))) {
      set_common(p.legacy, d, idx, !within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
      p.legacy_offset = d->offset_from_furthest; p.legacy_step = d->trajectory_point_step;
      p.legacy_use_yaw = d->use_path_orientations; p.legacy_max_ratio = d->max_path_occupancy_ratio;
      if (d->enabled && d->trajectory_point_step < 1) {return fail(h, MPPI_E_CONFIG, "PathAlignLegacyCritic.trajectory_point_step < 1");}
    }
    if (p.align.on && p.legacy.on && p.align_step != p.legacy_step) {
      return fail(h, MPPI_E_CONFIG, "PathAlignCritic and PathAlignLegacyCritic must share trajectory_point_step");
    }
    if (p.align.on || p.legacy.on) {
      p.sample_step = p.align.on ? p.align_step : p.legacy_step;
      p.n_samples = (p.T + p.sample_step - 1) / p.sample_step;
      p.sample_yaw = (p.align.on && p.align_use_yaw) || (p.legacy.on && p.legacy_use_yaw);
    }
    if ((d = find_kind(h, MPPI_CRITIC_PATH_ANGLE, &idx))) {
      set_common(p.angle, d, idx, !within_tolerance(d->threshold_to_consider, rx, ry, gx, gy));
      p.angle_offset = d->offset_from_furthest;
      // path_angle_critic.cpp:23-50
      const float vx_min = cfg.vx_min;
      bool reversing_allowed = true;
      if (fabs(vx_min) < 1e-6) {reversing_allowed = false;} else if (vx_min < 0.0) {reversing_allowed = true;}
      bool forward_preference = d->forward_preference != 0;
      if (!reversing_allowed) {forward_preference = true;}
      p.angle_reversing = reversing_allowed; p.angle_forward_pref = forward_preference;
      if (p.angle.on) {
        // path_angle_critic.cpp:79-83 for every index the furthest point could select.  The reference's test is
        // posePointAngle(...) < max_angle (atan2f + fmod per point: most of this function's time at 40 points).  With
        // forward_preference the angle A in [0, pi] is the one between the heading and the direction to the point, so
        // "A < max" is "cos A > cos max": decided from a dot product wherever that is further than 1e-5 from the
        // threshold (atan2f, the float roundings of the reference and the rounding of A to float move cos A by < 1e-6);
        // the reference's own arithmetic decides the rest, so the gate is the reference's gate bit for bit.
        const float thr = d->max_angle_to_furthest;
        const bool fast = forward_preference && thr > 1.0e-3f && thr < 3.1f;
        const float pose_xf = static_cast<float>(rx), pose_yf = static_cast<float>(ry), pose_yawf = static_cast<float>(in->pose_yaw);
        const double ch = std::cos(static_cast<double>(pose_yawf)), sh = std::sin(static_cast<double>(pose_yawf));
        const double ct = std::cos(static_cast<double>(thr));
        for (int j = 0; j < N; ++j) {
          const float gxj = in->path_x[j], gyj = in->path_y[j];
          int decided = -1;
          if (fast) {
            const double dxj = static_cast<double>(gxj - pose_xf), dyj = static_cast<double>(gyj - pose_yf);   // float differences, as atan2f gets them
            const double dd = dxj * dxj + dyj * dyj;
            if (dd > 1.0e-12) {
              const double c = (dxj * ch + dyj * sh) / std::sqrt(dd);
              if (c < ct - 1.0e-5) {decided = 1;} else if (c > ct + 1.0e-5) {decided = 0;}
            }
          }
          const bool open = decided >= 0 ? decided == 1 :
            !(pose_point_angle(rx, ry, in->pose_yaw, gxj, gyj, forward_preference) < thr);
          gate[j] = open ? 1 : 0;
          // only indices the critic can select count (furthest + offset_from_furthest, clamped): the point under the robot
          // (j = 0: atan2f(0, 0) = 0, i.e. the angle is the heading itself) must not force the trajectory spills
          any_gate_open = any_gate_open || (open && j >= std::max(0, std::min(p.angle_offset, N - 1)));
        }
      }
    }
  }
  // ---- everything K3 decides from the furthest reached path point alone, tabulated per candidate value f
  //      (the device only knows f after K2; path_follow_critic.cpp:45-58, path_align_critic.cpp:56-72,
  //       path_angle_critic.cpp:73-83)
  {
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
      unsigned char src = 0;
      switch (kind) {
        case MPPI_CRITIC_PATH_FOLLOW: src = p.follow.on ? 2 : 0; break;
        case MPPI_CRITIC_PATH_ALIGN: src = p.align.on ? 3 : 0; break;
        case MPPI_CRITIC_PATH_ALIGN_LEGACY: src = p.legacy.on ? 4 : 0; break;
        case MPPI_CRITIC_PATH_ANGLE: src = p.angle.on ? 5 : 0; break;
        case MPPI_CRITIC_CONSTRAINT: src = p.constraint.on ? 1 : 0; break;
        case MPPI_CRITIC_COST: src = p.cost.on ? 1 : 0; break;
        case MPPI_CRITIC_GOAL: src = p.goal.on ? 1 : 0; break;
        case MPPI_CRITIC_GOAL_ANGLE: src = p.goal_angle.on ? 1 : 0; break;
        case MPPI_CRITIC_OBSTACLES: src = p.obst.on ? 1 : 0; break;
        case MPPI_CRITIC_PREFER_FORWARD: src = p.forward.on ? 1 : 0; break;
        case MPPI_CRITIC_TWIRLING: src = p.twirl.on ? 1 : 0; break;
        case MPPI_CRITIC_VELOCITY_DEADBAND: src = p.deadband.on ? 1 : 0; break;
        default: break;
      }
      p.src_base[q] = src;
    }
    // first valid index at or after i (N if none)
    std::vector<int> & next_valid = h->scratch_next;
    next_valid.assign(N + 1, N);
    for (int i = N - 1; i >= 0; --i) {next_valid[i] = valid[i] ? i : next_valid[i + 1];}
    const int path_size = N - 1;
    auto align_gate = [&](int f, int offset, float max_ratio) -> bool {
        if (f < offset) {return false;}
        const int closest = p.closest_path_pt;
        const float range = static_cast<float>(static_cast<long long>(f) - closest);
        unsigned invalid_ctr = 0;
        if (f > closest) {invalid_ctr = static_cast<unsigned>(invalid_before[f]) - static_cast<unsigned>(invalid_before[closest]);}
        // the reference bails out of its counting loop as soon as ctr / range > ratio with ctr > 2; the count only
        // grows and the range is fixed, so the final count decides
        return !(invalid_ctr > 2 && static_cast<float>(invalid_ctr) / range > max_ratio);
      };
    for (int f = 0; f < N; ++f) {
      int fidx = std::min(f + p.follow_offset, path_size);
      if (fidx < path_size - 1) {fidx = std::min(next_valid[fidx], path_size - 1);}
      follow_tab[f] = static_cast<uint16_t>(std::max(fidx, 0));
      unsigned fl = 0;
      if (align_gate(f, p.align_offset, p.align_max_ratio) && f > 0) {fl |= 1u;}
      if (align_gate(f, p.legacy_offset, p.legacy_max_ratio) && (N - 1) >= 1) {fl |= 2u;}
      if (gate[std::min(f + p.angle_offset, N - 1)]) {fl |= 4u;}
      flags[f] = static_cast<uint8_t>(fl);
    }
  }
  p.spill_traj = ((h->want_mask & MPPI_WANT_TRAJECTORIES) || any_gate_open || mode == 1) ? 1 : 0;
  p.noise_tm = (h->stream_layout && mode == 0) ? 1 : 0;
  p.scan_mode = h->scan_mode;
  p.need_furthest = (p.follow.idx >= 0 || p.angle.idx >= 0 || p.align.idx >= 0 || p.legacy.idx >= 0) ? 1 : 0;
  h->last = p;
  return MPPI_OK;
}

// gridDim.y of weighted_sums_tm_kernel: enough row groups to put ~3 blocks on every SM, but at least one row per warp
int weighted_sums_row_groups(int T, int chunks)
{
  const int rows = 3 * T, warps = kWsThreads / 32;
  const int want = (3 * 148 + chunks - 1) / chunks;
  return std::max(1, std::min((rows + warps - 1) / warps, want));
}

int pick_segments(const mppi_handle * h)
{
  if (h->segments_override > 0) {return h->segments_override;}
  const int tiles = (h->B + kTile - 1) / kTile;
  int S = 8;
  if (tiles > 148 * 4) {S = 4;}
  while (S > 1 && S > h->T) {S >>= 1;}
  return S;
}

// TMA descriptors of the time-major noise planes [T + pad][B] for weighted_sums_tma_kernel: box = kPsRows rows x kPsBoxCols
// columns, no swizzle (a warp reads one row with 16-byte vectors at consecutive lanes: conflict free as it lies), columns
// beyond B are zero-filled by the TMA unit.  cuTensorMapEncodeTiled is a driver entry point; it is fetched through the
// runtime (cudaGetDriverEntryPoint), so the library still links against nothing but the static runtime.
bool make_noise_maps(mppi_handle * h)
{
  typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void * fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
      cudaGetLastError();
      return false;
    }
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  if (h->B % 4 != 0) {return false;}   // the row pitch must be a multiple of 16 bytes
  for (int i = 0; i < 3; ++i) {
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(h->B), static_cast<cuuint64_t>(h->T + kNoisePadRows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(h->B) * sizeof(float)};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(kPsBoxCols), static_cast<cuuint32_t>(kPsRows)};
    const cuuint32_t estr[2] = {1, 1};
    if (encode(&h->noise_map[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, h->d_noise[i], dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
      return false;
    }
  }
  return true;
}

DevBuffers make_bufs(mppi_handle * h, int mode)
{
  DevBuffers b;
  if (mode == 0) {
    b.in_a = h->d_noise[0]; b.in_b = h->d_noise[1]; b.in_c = h->d_noise[2];
    b.in_x = b.in_y = b.in_yaw = nullptr;
  } else {
    b.in_a = h->d_inj[0]; b.in_b = h->d_inj[1]; b.in_c = h->d_inj[2];
    b.in_x = h->d_inj[3]; b.in_y = h->d_inj[4]; b.in_yaw = h->d_inj[5];
  }
  b.cs = h->d_cs; b.crit_rows = h->d_crit_rows;
  b.samples_x = h->d_samples[0]; b.samples_y = h->d_samples[1]; b.samples_yaw = h->d_samples[2];
  b.end_xy = h->d_end_xy;
  b.spill_x = h->d_spill[0]; b.spill_y = h->d_spill[1]; b.spill_yaw = h->d_spill[2];
  b.spill_cells = h->d_cells;
  b.vis_xy = h->d_vis;
  b.costs = h->d_costs; b.partials = h->d_partials; b.rank_partial = h->d_rank_partial; b.out = h->d_out; b.st = h->d_st;
  for (int r = 0; r < kMaxRanks; ++r) {b.peer.box[r] = h->peer_mode ? h->peer_box[r] : nullptr;}
  b.peer.seq = h->d_seq;
  b.peer.rank = h->rank;
  b.peer.nranks = h->peer_mode ? h->nranks : 1;
  b.pk_up = h->d_pk;
  b.pk_x1 = h->d_pk ? h->d_pk + h->upd_blocks : nullptr;
  b.pk_rec = h->d_pk ? h->d_pk + 2 * h->upd_blocks : nullptr;
  b.pk_out = h->d_pk ? h->d_pk + static_cast<size_t>(h->upd_blocks) * (2 + 3 * h->T + 2) : nullptr;
  b.epoch = h->d_fepoch;
  // sticky "a bounded poll gave up" word in pinned host memory, behind the result packets (raise_comm_error)
  b.host_err = h->h_res ? reinterpret_cast<unsigned *>(h->h_res + 3 * static_cast<size_t>(h->T) + 9) : nullptr;
  static const int k3_fast = std::getenv("MPPI_K3_FAST") ? std::atoi(std::getenv("MPPI_K3_FAST")) : 1;   // measurement switch
  b.k3_fast = k3_fast;
  return b;
}

void drop_graphs(mppi_handle * h)
{
  for (auto & g : h->gexec) {
    if (g) {cudaGraphExecDestroy(g); g = nullptr;}
  }
}

constexpr int kFusedSmemMax = 226 * 1024;
constexpr size_t kZeroCopyMaxBytes = 96 * 1024;   // larger uploads (big costmaps) go through the copy engine

// validate + stage the costmap into pinned memory (the caller's buffer is only valid during the call: it holds
// the costmap mutex, controller.cpp:99-100); the async H2D copy itself is issued by enqueue_uploads
mppi_status stage_costmap(mppi_handle * h, const mppi_costmap & cm)
{
  const size_t bytes = static_cast<size_t>(cm.size_x) * cm.size_y;
  if (bytes == 0 || !cm.cells) {return fail(h, MPPI_E_CONFIG, "empty costmap");}
  if (!(cm.resolution > 0.0)) {return fail(h, MPPI_E_CONFIG, "costmap resolution must be > 0");}
  if (bytes > h->costmap_capacity && h->params_in_arena) {
    return fail(h, MPPI_E_CONFIG, "costmap larger than the slice of the bound group: mppi_batch_unbind first");
  }
  if (bytes > h->costmap_capacity) {
    // grow (outside the steady state: the costmap size only changes on reconfiguration); the record staged by
    // build_params moves with the buffer
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    drop_graphs(h);
    char * d_new = nullptr, * h_new = nullptr;
    CUDA_TRY(h, cudaMalloc(&d_new, kParamsCapacity + 256 + bytes));
    CUDA_TRY(h, cudaHostAlloc(&h_new, kParamsCapacity + 256 + bytes, cudaHostAllocMapped | cudaHostAllocPortable));
    std::memcpy(h_new, h->h_params, kParamsCapacity);
    CUDA_TRY(h, cudaMemcpy(d_new, h->d_params, kParamsCapacity, cudaMemcpyDeviceToDevice));
    cudaFree(h->d_params);
    cudaFreeHost(h->h_params);
    h->d_params = d_new; h->h_params = h_new;
    h->costmap_capacity = bytes;
  }
  const size_t off = (h->params_copy_bytes + 255) & ~static_cast<size_t>(255);
  h->d_costmap = reinterpret_cast<uint8_t *>(h->d_params + off);
  h->h_costmap = reinterpret_cast<uint8_t *>(h->h_params + off);
  h->costmap_bytes = bytes;
  // A costmap that lives in memory the caller registered as pinned is copied to the device from where it is (the
  // reference reads Costmap2D::getCharMap() in place, controller.cpp:99-100) - unless the upload is small enough for the
  // fused kernel to pull it out of the staging buffer itself, where the staging memcpy is the cheaper way.
  h->costmap_direct = nullptr;
  const bool small = !h->stream_layout && h->fused_enabled && h->zero_copy_enabled && h->nranks == 1 && off + bytes <= kZeroCopyMaxBytes;
  if (!small && !h->params_in_arena) {
    const char * c = reinterpret_cast<const char *>(cm.cells);
    for (const auto & r : h->pinned_ranges) {
      if (c >= r.first && c + bytes <= r.first + r.second) {h->costmap_direct = cm.cells; break;}
    }
  }
  if (!h->costmap_direct) {std::memcpy(h->h_costmap, cm.cells, bytes);}
  return MPPI_OK;
}

// bytes of [record | costmap], contiguous on both sides (stage_costmap)
size_t upload_bytes(const mppi_handle * h)
{
  return ((h->params_copy_bytes + 255) & ~static_cast<size_t>(255)) + h->costmap_bytes;
}

mppi_status enqueue_uploads(mppi_handle * h)
{
  if (h->costmap_direct) {
    // record from the staging buffer, costmap straight from the caller's registered memory (both complete before the
    // call returns: the result is ordered behind them on the stream)
    CUDA_TRY(h, cudaMemcpyAsync(h->d_params, h->h_params, h->params_copy_bytes, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_costmap, h->costmap_direct, h->costmap_bytes, cudaMemcpyHostToDevice, h->stream));
    return MPPI_OK;
  }
  CUDA_TRY(h, cudaMemcpyAsync(h->d_params, h->h_params, upload_bytes(h), cudaMemcpyHostToDevice, h->stream));
  return MPPI_OK;
}

// the exact set of features this cycle's record asks of the stream kernel (StreamFeature bits)
unsigned stream_feature_need(const DevParams & p)
{
  if (p.scan_mode != 0) {return SF_ALL;}   // the warp-scan experiment is compiled into the generic instance only
  unsigned need = 0;
  if (p.holonomic) {need |= SF_HOL;}
  if (p.model == MPPI_MODEL_ACKERMANN) {need |= SF_ACKER;}
  if (p.constraint.on) {need |= SF_CON;}
  if (p.forward.on) {need |= SF_FWD;}
  if (p.twirl.on) {need |= SF_TWIRL;}
  if (p.deadband.on) {need |= SF_DB;}
  if (p.goal.on) {need |= SF_GOAL;}
  if (p.goal_angle.on) {need |= SF_GANG;}
  if (p.cost.on) {need |= SF_COST;}
  if (p.obst.on) {need |= SF_OBST;}
  if ((p.cost.on && p.cost_fp) || (p.obst.on && p.obst_fp)) {need |= SF_FOOTPRINT;}
  if (p.want_cells || p.spill_traj || p.vis_b_step > 0) {need |= SF_SPILL;}
  return need;
}

// Compiled instances of the stream kernel.  The exact ones are straight-line code for one feature set (the deployed
// Omni critic list away from the goal, with and without footprint costs; the Obstacles-only benchmark config);
// anything else runs the generic instance, which tests the per-cycle flags at run time.
constexpr unsigned kSfOmniDefault = SF_HOL | SF_CON | SF_FWD | SF_TWIRL | SF_COST;
constexpr unsigned kSfOmniDefaultFp = kSfOmniDefault | SF_FOOTPRINT;
constexpr unsigned kSfObstaclesFp = SF_HOL | SF_OBST | SF_FOOTPRINT;

unsigned pick_stream_instance(unsigned need)
{
  if (need == kSfOmniDefault || need == kSfOmniDefaultFp || need == kSfObstaclesFp) {return need;}
  return SF_ALL;
}

int stream_block_threads(const mppi_handle * h)
{
  if (h->stream_threads_override > 0) {return h->stream_threads_override;}
  // fewer threads per block below ~4 full blocks per SM: same number of warps, spread evenly over the 148 SMs
  return h->B >= 148 * 4 * kStreamThreads ? kStreamThreads : 64;
}

template<unsigned F, bool kExact>
void launch_stream_instance(mppi_handle * h, int mode)
{
  const int nthr = stream_block_threads(h);
  const int Tp = ((h->T + kStreamChunk - 1) / kStreamChunk) * kStreamChunk;
  const size_t smem = kHotBytes + sizeof(float) * 3 * (Tp + nthr);   // hot record, control sequence, footprint slots
  rollout_score_stream_kernel<F, kExact><<<(h->B + nthr - 1) / nthr, nthr, smem, h->stream>>>(
    reinterpret_cast<const DevParams *>(h->d_params), h->d_costmap, make_bufs(h, mode));
}

mppi_status launch_regenerate(mppi_handle * h);


template<unsigned F, bool kExact>
cudaError_t fused_occupancy(int threads, size_t smem, int * blocks_per_sm)
{
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, tile_fused_kernel<F, kExact>, threads, smem);
}

// Stream layout, one rank, no evalControl tail: the merge kernel writes the result into pinned host memory as packets
// tagged with the epoch the path-cost kernel advanced (no D2H copy node, no stream synchronisation).
bool stream_packets(const mppi_handle * h)
{
  return h->stream_layout && h->nranks == 1 && h->tail_mode == 0 && h->d_fepoch != nullptr && h->packets_enabled;
}

// path capacity of the fused kernel's shared memory: rounded up to 64 points like the record copy (build_params), so that
// the captured graph survives small changes of the pruned path
int fused_path_capacity(const mppi_handle * h)
{
  return std::min(MPPI_MAX_PATH_POINTS, ((h->last.N + 63) / 64) * 64);
}

// sampled poses of PathAlign the fused kernel keeps scratch for (0 when the critic is not in the list)
int fused_align_samples(const mppi_handle * h)
{
  const DevParams & p = h->last;
  return (p.align.idx >= 0 && p.align_step >= 1) ? (h->T + p.align_step - 1) / p.align_step : 0;
}

// Does this cycle run as ONE cooperative launch of tile_fused_kernel?  Single rank, tile layout, and the whole grid
// co-resident (checked once per path size with the occupancy API; the generic instance is the largest one).
bool use_fused(mppi_handle * h)
{
  if (!h->fused_enabled || h->stream_layout || h->nranks > 1) {return false;}
  const int N = fused_path_capacity(h);
  const int key = N + 4096 * fused_align_samples(h);
  if (h->fused_key_N != key) {
    h->fused_key_N = key;
    h->fused_fits = false;
    const int S = pick_segments(h);
    const int grid = (h->B + kTile - 1) / kTile;
    const size_t smem = fused_smem_bytes(h->T, S, N, grid, fused_align_samples(h));
    int per_sm = 0;
    if (smem <= static_cast<size_t>(kFusedSmemMax) && fused_occupancy<SF_ALL, false>(kTile * S, smem, &per_sm) == cudaSuccess) {
      h->fused_fits = static_cast<long long>(per_sm) * h->num_sms >= grid;
    }
    cudaGetLastError();
  }
  return h->fused_fits;
}

template<unsigned F, bool kExact>
cudaError_t launch_fused_instance(mppi_handle * h, int iteration, uint2 * host_res, bool zero_copy, int tail_mode)
{
  const int S = pick_segments(h);
  const dim3 grid((h->B + kTile - 1) / kTile), block(kTile, S);
  int N = fused_path_capacity(h);
  const size_t smem = fused_smem_bytes(h->T, S, N, grid.x, fused_align_samples(h));
  const DevParams * dp = reinterpret_cast<const DevParams *>(h->d_params);
  const uint8_t * cm = h->d_costmap;
  DevBuffers bufs = make_bufs(h, 0);
  int B = h->B, T = h->T;
  // zero-copy upload: the kernel pulls [record | costmap] out of the pinned staging buffer itself (first iteration only)
  const uint4 * up_host = zero_copy ? reinterpret_cast<const uint4 *>(h->h_params) : nullptr;
  int up_vecs = zero_copy ? static_cast<int>((upload_bytes(h) + 15) / 16) : 0;
  float * hist = h->d_hist;
  void * args[] = {&dp, &cm, &bufs, &B, &T, &N, &iteration, &host_res, &up_host, &up_vecs, &tail_mode, &hist};
  if (!h->coop_launch) {   // experiment switch (MPPI_COOP=0): plain launch, no co-residency guarantee
    return cudaLaunchKernel(reinterpret_cast<const void *>(&tile_fused_kernel<F, kExact>), grid, block, args, smem, h->stream);
  }
  return cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(&tile_fused_kernel<F, kExact>), grid, block, args, smem, h->stream);
}

mppi_status launch_fused(mppi_handle * h, int iteration, uint2 * host_res, bool zero_copy, int tail_mode)
{
  cudaError_t e;
  switch (pick_stream_instance(stream_feature_need(h->last))) {
    case kSfOmniDefault: e = launch_fused_instance<kSfOmniDefault, true>(h, iteration, host_res, zero_copy, tail_mode); break;
    case kSfOmniDefaultFp: e = launch_fused_instance<kSfOmniDefaultFp, true>(h, iteration, host_res, zero_copy, tail_mode); break;
    case kSfObstaclesFp: e = launch_fused_instance<kSfObstaclesFp, true>(h, iteration, host_res, zero_copy, tail_mode); break;
    default: e = launch_fused_instance<SF_ALL, false>(h, iteration, host_res, zero_copy, tail_mode); break;
  }
  CUDA_TRY(h, e);
  h->launches++;
  return MPPI_OK;
}

mppi_status launch_rollout(mppi_handle * h, int mode)
{
  if (mode == 0 && h->stream_layout) {
    switch (pick_stream_instance(stream_feature_need(h->last))) {
      case kSfOmniDefault: launch_stream_instance<kSfOmniDefault, true>(h, mode); break;
      case kSfOmniDefaultFp: launch_stream_instance<kSfOmniDefaultFp, true>(h, mode); break;
      case kSfObstaclesFp: launch_stream_instance<kSfObstaclesFp, true>(h, mode); break;
      default: launch_stream_instance<SF_ALL, false>(h, mode); break;
    }
    CUDA_TRY(h, cudaGetLastError());
    h->launches++;
    return MPPI_OK;
  }
  const int S = pick_segments(h);
  const size_t smem = rollout_smem_bytes(h->T, S, mode);
  if (smem > 227 * 1024) {return fail(h, MPPI_E_CONFIG, "time_steps too large for the shared-memory tile");}
  const dim3 grid((h->B + kTile - 1) / kTile), block(kTile, S);
  const DevParams * dp = reinterpret_cast<const DevParams *>(h->d_params);
  const unsigned inst = mode == 0 ? pick_stream_instance(stream_feature_need(h->last)) : SF_ALL;
#define MPPI_LAUNCH_TILE(F, EXACT, MODE) \
  rollout_score_kernel<F, EXACT, MODE><<<grid, block, smem, h->stream>>>(dp, h->d_costmap, make_bufs(h, mode), h->B, h->T)
  if (mode == 1) {
    MPPI_LAUNCH_TILE(SF_ALL, false, 1);
  } else if (mode == 2) {
    MPPI_LAUNCH_TILE(SF_ALL, false, 2);
  } else if (inst == kSfOmniDefault) {
    MPPI_LAUNCH_TILE(kSfOmniDefault, true, 0);
  } else if (inst == kSfOmniDefaultFp) {
    MPPI_LAUNCH_TILE(kSfOmniDefaultFp, true, 0);
  } else if (inst == kSfObstaclesFp) {
    MPPI_LAUNCH_TILE(kSfObstaclesFp, true, 0);
  } else {
    MPPI_LAUNCH_TILE(SF_ALL, false, 0);
  }
#undef MPPI_LAUNCH_TILE
  CUDA_TRY(h, cudaGetLastError());
  h->launches++;
  return MPPI_OK;
}

// Launch with (pdl) or without programmatic stream serialisation: with it the kernel may start while its predecessor on
// the stream drains and synchronises inside (pdl_wait in mppi_kernels.cuh).  Captured into the cycle's CUDA graph like
// any other launch (programmatic dependency edge).
template<typename... KArgs, typename... Args>
cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args... args)
{
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// K3c of the stream layout: the TMA-fed kernel whenever the descriptors exist (B % 4 == 0), else the register-staged one
int weighted_sums_chunks(const mppi_handle * h)
{
  return h->ws_tma_ok ? (h->B + kPsChunk - 1) / kPsChunk : (h->B + kWsChunk - 1) / kWsChunk;
}

// the TMA-fed weighted-sums kernel merges, normalises and clips itself (no merge kernel behind it): single rank, and no
// coupling between the planes of a time step in the clip (Ackermann couples wz to vx).  Sharded over peer memory, exchange 2
// was tried in the same place (the last block of a row group pushing and polling its columns): 175 against 172 us per
// step at 2 GPUs - the exposed part is the last row group's merge plus the rank skew either way - and left out.
bool merge_in_weighted_sums(const mppi_handle * h)
{
  static const int enabled = std::getenv("MPPI_WS_MERGE") ? std::atoi(std::getenv("MPPI_WS_MERGE")) : 1;   // measurement switch
  return enabled && h->stream_layout && h->ws_tma_ok && h->nranks == 1 && h->cfg.motion_model != MPPI_MODEL_ACKERMANN && h->d_ws_done;
}

// host_res: the result leaves as packets (only looked at when the kernel merges itself)
mppi_status launch_weighted_sums(mppi_handle * h, uint2 * host_res = nullptr, bool allow_merge = false)
{
  const DevParams * dp = reinterpret_cast<const DevParams *>(h->d_params);
  const int chunks = weighted_sums_chunks(h);
  if (h->ws_tma_ok) {
    // row groups: every block pays the same start-up (1024 costs -> weights) before its first row, so few fat blocks beat
    // many thin ones: about 2.5 blocks per SM in all, never fewer than four row groups, at least two stages per block
    // (measured on B200 at 32768 ... 262144 x 100: 12 / 6 / 4 / 4 row groups; three times as many cost 7 - 13 us per step)
    const int stages = (holonomic(h) ? 3 : 2) * ((h->T + kPsRows - 1) / kPsRows);
    const int target = (5 * h->num_sms) / 2;
    const int gy = std::max(1, std::min(stages / 2, std::max(4, (target + chunks - 1) / chunks)));
    CUDA_TRY(h, launch_kernel(weighted_sums_tma_kernel, dim3(chunks, gy), dim3(kPsThreads), ps_smem_bytes(), h->stream, h->pdl_enabled,
      h->noise_map[0], h->noise_map[1], h->noise_map[2], dp, make_bufs(h, 0), h->T, h->B, holonomic(h) ? 1 : 0,
      (allow_merge && merge_in_weighted_sums(h)) ? h->d_ws_done : nullptr, host_res));
  } else {
    const int gy = weighted_sums_row_groups(h->T, chunks);
    CUDA_TRY(h, launch_kernel(weighted_sums_tm_kernel, dim3(chunks, gy), dim3(kWsThreads), 0, h->stream, h->pdl_enabled, dp, make_bufs(h, 0)));
  }
  CUDA_TRY(h, cudaGetLastError());
  h->launches++;
  return MPPI_OK;
}

mppi_status launch_update(mppi_handle * h, int mode, int iteration)
{
  if (mode == 0 && h->stream_layout) {
    // stream layout: totals + global minimum here, weights and weighted sums in weighted_sums_tm_kernel
    const int grid = std::min((h->B + kUpdThreads - 1) / kUpdThreads, 148 * 8);
    // the iteration that completes the result advances the packet epoch when the result leaves as packets
    const int bump = (stream_packets(h) && iteration + 1 == h->cfg.iteration_count) ? 1 : 0;
    // programmatic dependent launch behind the rollout kernel (not behind an NCCL all-reduce: that is a library launch)
    const bool pdl = h->pdl_enabled && !(h->nranks > 1 && !h->peer_mode);
    const DevParams * dp = reinterpret_cast<const DevParams *>(h->d_params);
    static const int k3a_blocks = std::getenv("MPPI_K3A_BLOCKS") ? std::atoi(std::getenv("MPPI_K3A_BLOCKS")) : 0;   // experiment
    if (k3a_blocks == 6) {
      CUDA_TRY(h, launch_kernel(path_costs_tm_kernel<6>, dim3(std::min(grid, 148 * 6)), dim3(kUpdThreads), k3_common_smem_bytes(), h->stream, pdl,
        dp, make_bufs(h, mode), iteration, bump));
    } else if (k3a_blocks == 4) {
      CUDA_TRY(h, launch_kernel(path_costs_tm_kernel<4>, dim3(std::min(grid, 148 * 4)), dim3(kUpdThreads), k3_common_smem_bytes(), h->stream, pdl,
        dp, make_bufs(h, mode), iteration, bump));
    } else if (h->B >= 131072 && k3a_blocks != 5) {
      CUDA_TRY(h, launch_kernel(path_costs_tm_kernel<8>, dim3(grid), dim3(kUpdThreads), k3_common_smem_bytes(), h->stream, pdl,
        dp, make_bufs(h, mode), iteration, bump));
    } else {
      CUDA_TRY(h, launch_kernel(path_costs_tm_kernel<5>, dim3(grid), dim3(kUpdThreads), k3_common_smem_bytes(), h->stream, pdl,
        dp, make_bufs(h, mode), iteration, bump));
    }
    CUDA_TRY(h, cudaGetLastError());
    h->launches++;
    return MPPI_OK;
  }
  path_softmax_update_kernel<<<h->upd_blocks, kUpdThreads, k3_tile_smem_bytes(h->T), h->stream>>>(
    reinterpret_cast<const DevParams *>(h->d_params), make_bufs(h, mode), h->nranks, iteration, h->B, h->T, mode);
  CUDA_TRY(h, cudaGetLastError());
  h->launches++;
  return MPPI_OK;
}

// device part of optimize(): iteration_count x {K2, [exchange 1], K3, [exchange 2, K4]} + D2H of the result, no sync
mppi_status enqueue_kernels(mppi_handle * h, bool prof)
{
  const int stride = 3 * h->T + 2;
  const bool fused = use_fused(h);
  for (int it = 0; it < h->cfg.iteration_count; ++it) {
    if (prof) {CUDA_TRY(h, cudaEventRecord(h->pev[0], h->stream));}
    if (fused) {
      // small batches: rollout, critics, softmax update and merge in one cooperative launch (pev: all of it counts as K2)
      // the launch that completes the result writes it to pinned host memory itself (packets) and, for
      // mppi_eval_control, runs the evalControl tail on tile 0
      const bool last = it + 1 == h->cfg.iteration_count;
      mppi_status s = launch_fused(h, it, last ? h->h_res : nullptr, h->zero_copy_now && it == 0, last ? h->tail_mode : 0);
      if (s != MPPI_OK) {return s;}
      if (prof) {
        CUDA_TRY(h, cudaEventRecord(h->pev[1], h->stream));
        CUDA_TRY(h, cudaEventRecord(h->pev[2], h->stream));
      }
      if (h->cfg.regenerate_noises && it + 1 < h->cfg.iteration_count) {
        if ((s = launch_regenerate(h)) != MPPI_OK) {return s;}
      }
      continue;
    }
    mppi_status s = launch_rollout(h, 0);
    if (s != MPPI_OK) {return s;}
    if (prof) {CUDA_TRY(h, cudaEventRecord(h->pev[1], h->stream));}
    if (h->nranks > 1 && !h->peer_mode) {
      // exchange 1: furthest path point candidate + "some trajectory survived" flags, one MAX all-reduce
      // (peer mode: the same exchange happens inside K3's preamble over the mapped mailboxes)
      NCCL_TRY(h, g_nccl.AllReduce(h->d_st, h->d_st, 1 + kMaxCritics, ncclUint32, ncclMax, h->comm, h->stream));
    }
    s = launch_update(h, 0, it);
    if (s != MPPI_OK) {return s;}
    const bool many = h->upd_blocks > kLastBlockMergeMax;
    const int merge_grid = (h->T + kMergeT - 1) / kMergeT;
    const DevParams * dp = reinterpret_cast<const DevParams *>(h->d_params);
    const int chunks = weighted_sums_chunks(h);
    if (h->stream_layout) {
      // K3 published costs + global minimum; weights and weighted control sums over the time-major noise
      const mppi_status ws = launch_weighted_sums(h, (stream_packets(h) && it + 1 == h->cfg.iteration_count) ? h->h_res : nullptr, true);
      if (ws != MPPI_OK) {return ws;}
    }
    if (h->nranks > 1 && h->peer_mode) {
      // exchange 2 over peer memory, fused with the local merge before it and the cross-rank merge after it
      if (prof) {CUDA_TRY(h, cudaEventRecord(h->pev[2], h->stream));}
      const bool merged_in_k3 = !h->stream_layout && !many;   // K3's last block already merged into rank_partial
      CUDA_TRY(h, launch_kernel(merge_exchange_finalize_kernel, dim3(merge_grid), dim3(kUpdThreads), 0, h->stream,
        h->pdl_enabled && h->stream_layout, dp, merged_in_k3 ? h->d_rank_partial : h->d_partials,
        merged_in_k3 ? 1 : (h->stream_layout ? chunks : h->upd_blocks), stride, make_bufs(h, 0)));
      CUDA_TRY(h, cudaGetLastError());
      h->launches++;
    } else {
      if (merge_in_weighted_sums(h)) {
        // nothing to launch: the weighted-sums kernel's last block per row group merged, clipped and delivered
      } else if (h->stream_layout || many) {
        // too many partial records for a serial merge in K3's last block (or the stream layout): merge in parallel
        CUDA_TRY(h, launch_kernel(merge_finalize_kernel, dim3(merge_grid), dim3(kUpdThreads), 0, h->stream, h->pdl_enabled && h->stream_layout,
          dp, h->d_partials, h->stream_layout ? chunks : h->upd_blocks, stride, make_bufs(h, 0), h->nranks > 1 ? 0 : 1, h->d_rank_partial,
          (stream_packets(h) && it + 1 == h->cfg.iteration_count) ? h->h_res : nullptr));
        CUDA_TRY(h, cudaGetLastError());
        h->launches++;
      }
      if (prof) {CUDA_TRY(h, cudaEventRecord(h->pev[2], h->stream));}
      if (h->nranks > 1) {
        // exchange 2: per-rank (min, sum, weighted control sums); merged redundantly on every rank
        NCCL_TRY(h, g_nccl.AllGather(h->d_rank_partial, h->d_gathered, stride, ncclFloat32, h->comm, h->stream));
        merge_finalize_kernel<<<merge_grid, kUpdThreads, 0, h->stream>>>(dp, h->d_gathered, h->nranks, stride, make_bufs(h, 0), 1, nullptr, nullptr);
        CUDA_TRY(h, cudaGetLastError());
        h->launches++;
      }
    }
    if (h->cfg.regenerate_noises && it + 1 < h->cfg.iteration_count) {
      if ((s = launch_regenerate(h)) != MPPI_OK) {return s;}
    }
  }
  if (h->tail_mode && !fused) {
    // evalControl's tail (Savitzky-Golay filter, command extraction, shift) stays on the device (the fused kernel runs it
    // itself)
    eval_tail_kernel<<<1, 32, 0, h->stream>>>(h->d_cs, h->d_hist, h->d_out, h->T, holonomic(h) ? 1 : 0, h->tail_mode == 2 ? 1 : 0);
    CUDA_TRY(h, cudaGetLastError());
    h->launches++;
  }
  if (prof) {CUDA_TRY(h, cudaEventRecord(h->pev[3], h->stream));}
  if (!fused && !stream_packets(h)) {
    CUDA_TRY(h, cudaMemcpyAsync(h->h_out, h->d_out, sizeof(float) * (3 * h->T + 6), cudaMemcpyDeviceToHost, h->stream));
  }
  if (h->cfg.regenerate_noises) {
    // the result is complete here; the redraw for the next cycle runs behind it, off the caller's critical path
    if (h->capturing) {
      CUDA_TRY(h, cudaEventRecordWithFlags(h->ev_result, h->stream, cudaEventRecordExternal));
    } else {
      CUDA_TRY(h, cudaEventRecord(h->ev_result, h->stream));
    }
    return launch_regenerate(h);
  }
  return MPPI_OK;
}

// One cycle on the handle's stream: [uploads], kernels, result copy; bracketed by ev0 / ev1.  The steady state
// (single rank, no per-kernel profiling) replays a captured CUDA graph: one launch instead of five.
mppi_status enqueue_optimize_impl(mppi_handle * h, bool with_upload);

// The host mirrors the device's packet epoch (fepoch_host) and advances it when a cycle is enqueued.  If enqueueing fails
// half-way, or a cycle ends with an error, the mirror is re-read from the device once the stream has drained: otherwise
// every later cycle would wait for a tag that is never written.
void resync_packet_epoch(mppi_handle * h)
{
  if (!h->d_fepoch) {return;}
  cudaStreamSynchronize(h->stream);
  uint32_t e = h->fepoch_host;
  if (cudaMemcpy(&e, h->d_fepoch, sizeof(uint32_t), cudaMemcpyDeviceToHost) == cudaSuccess) {h->fepoch_host = e;}
  cudaGetLastError();
}

mppi_status enqueue_optimize(mppi_handle * h, bool with_upload)
{
  const mppi_status s = enqueue_optimize_impl(h, with_upload);
  if (s != MPPI_OK && h->wait_packets) {
    const std::string keep = h->err;
    resync_packet_epoch(h);
    h->wait_packets = false;
    h->err = keep;
  }
  return s;
}

mppi_status enqueue_optimize_impl(mppi_handle * h, bool with_upload)
{
  const bool prof = h->profiling && h->cfg.iteration_count == 1;
  const bool graph_ok = h->use_graph && !prof && (h->nranks == 1 || h->peer_mode);   // NCCL calls are not captured
  h->ev_src = nullptr;
  const bool fused_now = use_fused(h);
  h->wait_packets = fused_now || stream_packets(h);
  h->zero_copy_now = with_upload && fused_now && h->zero_copy_enabled && upload_bytes(h) <= kZeroCopyMaxBytes;
  if (h->wait_packets) {
    // the fused kernel advances the epoch once per launch, the stream layout once per cycle
    h->fepoch_host += fused_now ? static_cast<uint32_t>(h->cfg.iteration_count) : 1u;
    h->result_tag = h->fepoch_host;
  }
  h->d2h_bytes = h->wait_packets ? sizeof(uint2) * (3 * h->T + 2 + (h->tail_mode ? 3 : 0)) : sizeof(float) * (3 * h->T + 6);
  // zero-copy: every tile also reads the hot part of the record over PCIe
  h->h2d_bytes = with_upload ? upload_bytes(h) + (h->zero_copy_now ? static_cast<size_t>(h->upd_blocks) * kHotBytes : 0) : 0;
  const uint64_t t_a = now_ns();
  bool ev0_recorded = false;
  if (h->timing && !graph_ok) {CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream)); ev0_recorded = true;}
  const uint64_t t_b = now_ns();
  h->host_ns[2] += t_b - t_a;
  if (graph_ok) {
    // the upload stays OUT of the graph: a copy node in a captured graph measured ~8 us slower than the same
    // cudaMemcpyAsync issued on the stream in front of the graph launch (profiles/, host phases)
    // Small uploads behind the fused kernel are not copied at all: the kernel reads the pinned staging buffer
    // (zero_copy_now, slot 1); the copy engine -> kernel hand-over alone costs more than the PCIe reads.
    if (with_upload && !h->zero_copy_now) {
      const mppi_status us = enqueue_uploads(h);
      if (us != MPPI_OK) {return us;}
      with_upload = false;
    }
    const int slot = (with_upload ? 1 : 0) + 2 * h->tail_mode + (h->timing ? 6 : 0);
    const unsigned inst = pick_stream_instance(stream_feature_need(h->last));   // the K2 instance is baked into the graph
    const int fkey = fused_now ? h->fused_key_N : -1;
    if (h->gexec[slot] && (h->gkey_params[slot] != h->params_copy_bytes || h->gkey_costmap[slot] != h->costmap_bytes ||
      h->gkey_inst[slot] != inst || h->gkey_fused[slot] != fkey))
    {
      cudaGraphExecDestroy(h->gexec[slot]);
      h->gexec[slot] = nullptr;
    }
    if (!h->gexec[slot]) {
      cudaGraph_t graph = nullptr;
      const uint64_t launches_before = h->launches;
      CUDA_TRY(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
      h->capturing = true;
      mppi_status s = MPPI_OK;
      // (external event nodes: the host reads them back after the launch)
      if (h->timing && cudaEventRecordWithFlags(h->ev0, h->stream, cudaEventRecordExternal) != cudaSuccess) {s = MPPI_E_CUDA;}
      if (s == MPPI_OK && with_upload && !h->zero_copy_now) {s = enqueue_uploads(h);}
      if (s == MPPI_OK) {s = enqueue_kernels(h, false);}
      if (s == MPPI_OK && h->timing && cudaEventRecordWithFlags(h->ev1, h->stream, cudaEventRecordExternal) != cudaSuccess) {s = MPPI_E_CUDA;}
      h->capturing = false;
      const cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
      h->launches = launches_before;   // capture launched nothing
      if (s != MPPI_OK || ce != cudaSuccess || !graph) {
        if (graph) {cudaGraphDestroy(graph);}
        cudaGetLastError();
        h->use_graph = false;            // fall back to plain stream launches for this handle
      } else {
        const cudaError_t ie = cudaGraphInstantiate(&h->gexec[slot], graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) {cudaGetLastError(); h->gexec[slot] = nullptr; h->use_graph = false;}
        h->gkey_params[slot] = h->params_copy_bytes;
        h->gkey_costmap[slot] = h->costmap_bytes;
        h->gkey_inst[slot] = inst;
        h->gkey_fused[slot] = fkey;
      }
    }
    if (h->gexec[slot]) {
      CUDA_TRY(h, cudaGraphLaunch(h->gexec[slot], h->stream));
      const uint64_t t_c = now_ns();
      h->host_ns[3] += t_c - t_b;
      h->launches += (use_fused(h) ? 1ull : (h->stream_layout ? 4ull : (h->upd_blocks > kLastBlockMergeMax ? 3ull : 2ull))) *
        h->cfg.iteration_count + (h->tail_mode && !use_fused(h) ? 1ull : 0ull);
      h->host_ns[4] += now_ns() - t_c;
      return MPPI_OK;
    }
  }
  if (h->timing && !ev0_recorded) {CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));}
  mppi_status s = MPPI_OK;
  if (with_upload && !h->zero_copy_now) {s = enqueue_uploads(h);}
  if (s != MPPI_OK) {return s;}
  if ((s = enqueue_kernels(h, prof)) != MPPI_OK) {return s;}
  if (h->timing) {CUDA_TRY(h, cudaEventRecord(h->ev1, h->stream));}
  return MPPI_OK;
}

// The fused kernel (or the tail kernel behind it) writes the result straight into pinned host memory as packets
// {value, tag}; a packet whose tag is the tag of the last launch enqueued is complete.  Polling them replaces the D2H
// copy node and the stream synchronisation.  The stream is queried every few thousand polls so that a failed launch
// surfaces as an error instead of a hang.
mppi_status wait_result_packets(mppi_handle * h)
{
  const int n = 3 * h->T + 2 + (h->tail_mode ? 3 : 0);
  const uint32_t tag = h->result_tag;
  const uint64_t * pk = reinterpret_cast<const uint64_t *>(h->h_res);
  uint32_t * dst = reinterpret_cast<uint32_t *>(h->h_out);
  uint64_t spins = 0;
  bool drained = false;
  for (int i = 0; i < n; ++i) {
    for (;;) {
      const uint64_t v = __atomic_load_n(pk + i, __ATOMIC_ACQUIRE);
      if (static_cast<uint32_t>(v >> 32) == tag) {dst[i] = static_cast<uint32_t>(v); break;}
      if ((++spins & 4095u) == 0u) {
        if (drained) {
          // everything enqueued has run and the packet is still missing: resynchronise the epoch mirror and report
          cudaMemcpy(&h->fepoch_host, h->d_fepoch, sizeof(uint32_t), cudaMemcpyDeviceToHost);
          return fail(h, MPPI_E_CUDA, "fused kernel finished without delivering its result packets");
        }
        const cudaError_t q = cudaStreamQuery(h->stream);
        if (q == cudaSuccess) {
          drained = true;
        } else if (q != cudaErrorNotReady) {
          return fail(h, MPPI_E_CUDA, std::string("cudaStreamQuery: ") + cudaGetErrorString(q));
        }
      }
#if defined(__x86_64__) || defined(__i386__)
      __builtin_ia32_pause();
#endif
    }
  }
  return MPPI_OK;
}

mppi_status finish_optimize(mppi_handle * h, mppi_cycle_out * out)
{
  const uint64_t t_a = now_ns();
  if (h->cfg.regenerate_noises) {
    h->noise_stream += static_cast<uint64_t>(h->cfg.iteration_count);   // host mirror of d_epoch
  }
  if (h->wait_packets) {
    mppi_status ws = wait_result_packets(h);
    if (ws != MPPI_OK) {return ws;}
    // a tile gave up waiting for another tile's packets (raise_comm_error): the result above is not to be trusted
    volatile unsigned * host_err = reinterpret_cast<volatile unsigned *>(h->h_res + 3 * static_cast<size_t>(h->T) + 9);
    if (*host_err != 0u) {
      *host_err = 0u;
      resync_packet_epoch(h);
      cudaMemsetAsync(&h->d_st->comm_error, 0, sizeof(unsigned), h->stream);
      return fail(h, h->nranks > 1 ? MPPI_E_NCCL : MPPI_E_CUDA,
               "an in-kernel packet exchange timed out (a tile or rank never delivered): result discarded");
    }
    if (h->timing) {CUDA_TRY(h, cudaEventSynchronize(h->cfg.regenerate_noises ? h->ev_result : (h->ev_src ? h->ev_src : h)->ev1));}
  } else if (h->cfg.regenerate_noises) {
    CUDA_TRY(h, cudaEventSynchronize(h->ev_result));
  } else {
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  }
  const uint64_t t_b = now_ns();
  h->host_ns[5] += t_b - t_a;
  const int T = h->T;
  h->spilled_traj = h->last.spill_traj != 0;
  h->spilled_cells = h->last.want_cells != 0;
  h->vis_valid = h->last.vis_b_step > 0;
  h->have_rows = true;
  if (out) {
    if (out->control_vx) {std::memcpy(out->control_vx, h->h_out, sizeof(float) * T);}
    if (out->control_vy) {std::memcpy(out->control_vy, h->h_out + T, sizeof(float) * T);}
    if (out->control_wz) {std::memcpy(out->control_wz, h->h_out + 2 * T, sizeof(float) * T);}
    int32_t ff;
    uint32_t fu;
    std::memcpy(&ff, h->h_out + 3 * T, 4);
    std::memcpy(&fu, h->h_out + 3 * T + 1, 4);
    out->fail_flag = ff;
    out->furthest_reached_path_point = fu;
  }
  // device time of the cycle (events around everything enqueued for it), only when asked for: reading two events back
  // costs several microseconds of host time
  float ms = 0.0f;
  if (h->timing) {
    const mppi_handle * es = h->ev_src ? h->ev_src : h;
    cudaEventElapsedTime(&ms, es->ev0, h->cfg.regenerate_noises ? h->ev_result : es->ev1);
  }
  h->prof_ms[3] = ms;
  if (out) {out->device_ms = ms;}
  if (h->peer_mode) {
    uint32_t comm_error;
    std::memcpy(&comm_error, h->h_out + 3 * T + 5, 4);
    if (comm_error) {return fail(h, MPPI_E_NCCL, "peer-memory exchange timed out: a rank did not arrive");}
  }
  if (h->profiling && h->cfg.iteration_count == 1) {
    cudaEventElapsedTime(&h->prof_ms[0], h->pev[0], h->pev[1]);
    // with sharding the span pev[1]..pev[2] also holds exchange 1; K3 alone is not separable there
    cudaEventElapsedTime(&h->prof_ms[1], h->pev[1], h->pev[2]);
    cudaEventElapsedTime(&h->prof_ms[2], h->pev[2], h->pev[3]);
    if (use_fused(h)) {h->prof_ms[1] = 0.0f; h->prof_ms[2] = 0.0f;}   // fused kernel: everything is in [0]
  }
  h->host_ns[6] += now_ns() - t_b;
  h->host_ns[7] += 1;
  return MPPI_OK;
}

// room for `records` softmax records in d_gathered (grown outside the steady state: the shard count changes on reconfiguration)
mppi_status ensure_gathered(mppi_handle * h, int records)
{
  if (h->d_gathered && h->gathered_capacity >= static_cast<size_t>(records)) {return MPPI_OK;}
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (h->d_gathered) {cudaFree(h->d_gathered); h->d_gathered = nullptr; h->gathered_capacity = 0;}
  const size_t cap = static_cast<size_t>(std::max(records, 8));
  CUDA_TRY(h, cudaMalloc(&h->d_gathered, cap * (3 * static_cast<size_t>(h->T) + 2) * sizeof(float)));
  h->gathered_capacity = cap;
  return MPPI_OK;
}

mppi_status ensure_injection_buffers(mppi_handle * h)
{
  const size_t n = static_cast<size_t>(h->B) * h->T * sizeof(float);
  for (int i = 0; i < 6; ++i) {
    if (!h->d_inj[i]) {CUDA_TRY(h, cudaMalloc(&h->d_inj[i], n));}
  }
  return MPPI_OK;
}
mppi_status ensure_tmp(mppi_handle * h)
{
  if (!h->d_tmp) {CUDA_TRY(h, cudaMalloc(&h->d_tmp, static_cast<size_t>(h->B) * h->T * sizeof(float)));}
  return MPPI_OK;
}

template<typename V>
mppi_status fetch_time_major(mppi_handle * h, const V * d_src, V * host_dst)
{
  mppi_status s = ensure_tmp(h);
  if (s != MPPI_OK) {return s;}
  const dim3 grid((h->B + 31) / 32, (h->T + 31) / 32), block(32, 8);
  transpose_tb_to_bt_kernel<V><<<grid, block, 0, h->stream>>>(d_src, reinterpret_cast<V *>(h->d_tmp), h->T, h->B);
  CUDA_TRY(h, cudaGetLastError());
  CUDA_TRY(h, cudaMemcpyAsync(host_dst, h->d_tmp, static_cast<size_t>(h->B) * h->T * sizeof(V), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status sync_epoch(mppi_handle * h)
{
  const unsigned long long e = h->noise_stream;
  CUDA_TRY(h, cudaMemcpyAsync(h->d_epoch, &e, sizeof(e), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

// regenerate_noises (noise_generator.cpp:54-63,97-105): redraw the noise once the current set has been consumed.  The
// stream index comes from device memory (d_epoch) so that a captured graph draws a new set at every replay.
mppi_status launch_regenerate(mppi_handle * h)
{
  const long long total = static_cast<long long>(h->B) * ((h->T + 3) / 4);
  const int blocks = static_cast<int>(std::min<long long>((total + 255) / 256, 148LL * 16));
  noise_philox_kernel<<<std::max(blocks, 1), 256, 0, h->stream>>>(
    h->d_noise[0], h->d_noise[1], h->d_noise[2], h->B, h->T, h->cfg.vx_std, h->cfg.vy_std, h->cfg.wz_std,
    holonomic(h) ? 1 : 0, h->cfg.seed, 0, static_cast<uint64_t>(h->cfg.shard_offset), h->stream_layout ? 1 : 0, h->d_epoch);
  advance_epoch_kernel<<<1, 1, 0, h->stream>>>(h->d_epoch);
  CUDA_TRY(h, cudaGetLastError());
  h->launches += 2;
  return MPPI_OK;
}

mppi_status do_reset(mppi_handle * h)
{
  const size_t T = h->T, B = h->B;
  h->cur = h->base;
  CUDA_TRY(h, cudaMemsetAsync(h->d_cs, 0, 3 * T * sizeof(float), h->stream));
  CUDA_TRY(h, cudaMemsetAsync(h->d_hist, 0, 12 * sizeof(float), h->stream));   // control_history_ (optimizer.cpp:120-123)
  CUDA_TRY(h, cudaMemsetAsync(h->d_costs, 0, B * sizeof(float), h->stream));
  CUDA_TRY(h, cudaMemsetAsync(h->d_st, 0, sizeof(DevState), h->stream));
  // NoiseGenerator::reset (noise_generator.cpp:76-95): redraw
  const int threads = 256;
  const long long total = static_cast<long long>(B) * ((T + 3) / 4);
  const int blocks = static_cast<int>(std::min<long long>((total + threads - 1) / threads, 148LL * 16));
  noise_philox_kernel<<<std::max(blocks, 1), threads, 0, h->stream>>>(
    h->d_noise[0], h->d_noise[1], h->d_noise[2], h->B, h->T, h->cfg.vx_std, h->cfg.vy_std, h->cfg.wz_std,
    holonomic(h) ? 1 : 0, h->cfg.seed, h->noise_stream, static_cast<uint64_t>(h->cfg.shard_offset), h->stream_layout ? 1 : 0, nullptr);
  CUDA_TRY(h, cudaGetLastError());
  h->launches++;
  h->noise_stream++;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->cycle_uploaded = false;
  return sync_epoch(h);
}

// ---- multi-robot batch -----------------------------------------------------------------------------
void batch_unbind_group(mppi_handle * leader)
{
  if (!leader) {return;}
  cudaSetDevice(leader->device);
  cudaStreamSynchronize(leader->stream);
  if (leader->copy_stream) {
    cudaStreamSynchronize(leader->copy_stream);
    cudaStreamDestroy(leader->copy_stream);
    leader->copy_stream = nullptr;
    for (auto & e : leader->ev_upload) {if (e) {cudaEventDestroy(e); e = nullptr;}}
  }
  std::vector<mppi_handle *> group = leader->batch_group;
  for (mppi_handle * m : group) {
    if (m != leader && m->own_stream) {m->stream = m->own_stream; m->own_stream = nullptr;}
    m->batch_leader = nullptr;
    m->ev_src = nullptr;
    drop_graphs(m);
    if (m->params_in_arena) {
      // back to buffers of its own (the staged cycle does not survive: the next call uploads again)
      const size_t bytes = kParamsCapacity + 256 + m->costmap_capacity;
      m->h_params = nullptr; m->d_params = nullptr;
      cudaHostAlloc(&m->h_params, bytes, cudaHostAllocMapped | cudaHostAllocPortable);
      cudaMalloc(&m->d_params, bytes);
      m->d_costmap = nullptr; m->h_costmap = nullptr;
      m->params_in_arena = false;
      m->cycle_uploaded = false;
    }
    if (m->h_res) {std::memset(m->h_res, 0, (3 * static_cast<size_t>(m->T) + 10) * sizeof(uint2));}   // tags of the group era
  }
  if (leader->arena_h) {cudaFreeHost(leader->arena_h); leader->arena_h = nullptr;}
  if (leader->arena_d) {cudaFree(leader->arena_d); leader->arena_d = nullptr;}
  leader->arena_slice = 0;
  leader->batch_mode = 0;
  leader->batch_group.clear();
  leader->jobs_sent.clear();
  if (leader->h_jobs) {cudaFreeHost(leader->h_jobs); leader->h_jobs = nullptr;}
  if (leader->d_jobs) {cudaFree(leader->d_jobs); leader->d_jobs = nullptr;}
  if (leader->d_ticket) {cudaFree(leader->d_ticket); leader->d_ticket = nullptr;}
  leader->ticket_base = 0;
}

// is hs[0..n) exactly a bound group, in bind order?
bool batch_is_group(mppi_handle ** hs, int n)
{
  if (n < 2 || !hs[0] || hs[0]->batch_leader != hs[0] || static_cast<int>(hs[0]->batch_group.size()) != n) {return false;}
  for (int i = 0; i < n; ++i) {
    if (hs[i] != hs[0]->batch_group[i]) {return false;}
  }
  return true;
}

constexpr int kBatchChunk = 16;   // robots per launch: the host prepares the next chunk's records while this one runs

template<unsigned F, bool kExact>
cudaError_t launch_batch_instance(mppi_handle * leader, int c0, int n, int G, dim3 block, size_t smem)
{
  tile_fused_batch_kernel<F, kExact><<<dim3(static_cast<unsigned>(n) * G), block, smem, leader->stream>>>(
    leader->d_jobs + c0, G, leader->d_ticket, leader->ticket_base);
  return cudaGetLastError();
}

// One launch for the members [c0, c0 + n) of a bound group (their records are built, uploads staged).  Returns
// MPPI_E_STATE without having launched anything when they do not qualify this cycle: the caller then runs them one by
// one (they share a stream, so that is correct, only slower).  `first` / `last`: this is the first / last chunk of the
// call (the leader's events bracket the whole call).
mppi_status batch_launch(mppi_handle * L, mppi_handle ** hs, int c0, int n, bool with_upload, bool first, bool last)
{
  // the exact instance when every member asks for the same one, else the generic instance (it tests the per-cycle flags)
  unsigned inst = pick_stream_instance(stream_feature_need(hs[0]->last));
  for (int i = 1; i < n; ++i) {
    if (pick_stream_instance(stream_feature_need(hs[i]->last)) != inst) {inst = SF_ALL; break;}
  }
  const int S = pick_segments(L);
  const int G = (L->B + kTile - 1) / kTile;
  const int n_cap = fused_path_capacity(hs[0]), n_s = fused_align_samples(hs[0]);
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    const char * why = nullptr;
    if (!use_fused(h)) {why = "fused kernel not applicable";}
    else if (h->tail_mode != 0 || h->cfg.iteration_count != 1 || h->profiling) {why = "tail / iteration_count / profiling";}
    else if (fused_path_capacity(h) != n_cap || fused_align_samples(h) != n_s) {why = "different path capacity / PathAlign samples";}
    if (why) {
      L->err = std::string("batched launch not used: member ") + std::to_string(c0 + i) + ": " + why;
      return MPPI_E_STATE;
    }
  }
  const size_t smem = fused_smem_bytes(L->T, S, n_cap, G, n_s);
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    h->wait_packets = true;
    h->ev_src = L;
    h->zero_copy_now = with_upload && h->zero_copy_enabled && upload_bytes(h) <= kZeroCopyMaxBytes;
    if (with_upload && !h->zero_copy_now) {
      const mppi_status us = enqueue_uploads(h);
      if (us != MPPI_OK) {return us;}
    }
    FusedJob & j = L->h_jobs[c0 + i];
    std::memset(&j, 0, sizeof(j));
    j.Pg = reinterpret_cast<const DevParams *>(h->d_params);
    j.cm = h->d_costmap;
    j.bufs = make_bufs(h, 0);
    j.B = h->B; j.T = h->T; j.n_cap = n_cap; j.iteration = 0;
    j.host_res = h->h_res;
    j.up_host = h->zero_copy_now ? reinterpret_cast<const uint4 *>(h->h_params) : nullptr;
    j.up_vecs = h->zero_copy_now ? static_cast<int>((upload_bytes(h) + 15) / 16) : 0;
  }
  // the device copy of the job table is re-sent only where it changed (pointers and sizes are the same every cycle)
  const size_t off = sizeof(FusedJob) * static_cast<size_t>(c0), bytes = sizeof(FusedJob) * static_cast<size_t>(n);
  if (std::memcmp(L->jobs_sent.data() + off, L->h_jobs + c0, bytes) != 0) {
    CUDA_TRY(L, cudaMemcpyAsync(L->d_jobs + c0, L->h_jobs + c0, bytes, cudaMemcpyHostToDevice, L->stream));
    std::memcpy(L->jobs_sent.data() + off, L->h_jobs + c0, bytes);
  }
  if (first && L->timing) {CUDA_TRY(L, cudaEventRecord(L->ev0, L->stream));}
  const dim3 block(kTile, S);
  cudaError_t e;
  switch (inst) {
    case kSfOmniDefault: e = launch_batch_instance<kSfOmniDefault, true>(L, c0, n, G, block, smem); break;
    case kSfOmniDefaultFp: e = launch_batch_instance<kSfOmniDefaultFp, true>(L, c0, n, G, block, smem); break;
    case kSfObstaclesFp: e = launch_batch_instance<kSfObstaclesFp, true>(L, c0, n, G, block, smem); break;
    default: e = launch_batch_instance<SF_ALL, false>(L, c0, n, G, block, smem); break;
  }
  CUDA_TRY(L, e);
  if (last && L->timing) {CUDA_TRY(L, cudaEventRecord(L->ev1, L->stream));}
  L->ticket_base += static_cast<uint32_t>(n) * static_cast<uint32_t>(G);
  L->launches++;
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    h->fepoch_host += 1u;
    h->result_tag = h->fepoch_host;
    h->d2h_bytes = sizeof(uint2) * (3 * h->T + 2);
    h->h2d_bytes = with_upload ? upload_bytes(h) + (h->zero_copy_now ? static_cast<size_t>(h->upd_blocks) * kHotBytes : 0) : 0;
  }
  return MPPI_OK;
}

// ---- mode 2: the group in the stream layout, four batched kernels for all robots -------------------------------
// [B][T] -> [T][B] for the three noise planes of a handle that was created in the tile layout
mppi_status to_stream_layout(mppi_handle * h)
{
  if (h->stream_layout) {return MPPI_OK;}
  if ((static_cast<unsigned long long>(h->T) + kNoisePadRows) * static_cast<unsigned long long>(h->B) >= (1ull << 32)) {
    return fail(h, MPPI_E_CONFIG, "batch_size * time_steps too large for the 32-bit offsets of the stream layout");
  }
  mppi_status s = ensure_tmp(h);
  if (s != MPPI_OK) {return s;}
  const size_t plane = static_cast<size_t>(h->B) * h->T * sizeof(float);
  const dim3 grid((h->T + 31) / 32, (h->B + 31) / 32), block(32, 8);
  for (int i = 0; i < 3; ++i) {
    CUDA_TRY(h, cudaMemcpyAsync(h->d_tmp, h->d_noise[i], plane, cudaMemcpyDeviceToDevice, h->stream));
    transpose_tb_to_bt_kernel<float><<<grid, block, 0, h->stream>>>(h->d_tmp, h->d_noise[i], h->B, h->T);
    CUDA_TRY(h, cudaGetLastError());
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  drop_graphs(h);
  h->stream_layout = true;
  h->fused_key_N = -1;
  return MPPI_OK;
}

constexpr int kStreamBatchChunk = 64;   // robots per upload + four launches: the host builds the next chunk's records meanwhile

template<unsigned F, bool kExact>
cudaError_t launch_stream_batch_instance(mppi_handle * L, const FusedJob * jobs, int n, int nthr, size_t smem)
{
  rollout_score_stream_batch_kernel<F, kExact><<<dim3((L->B + nthr - 1) / nthr, n), nthr, smem, L->stream>>>(jobs);
  return cudaGetLastError();
}

// does every member qualify for the batched stream launch this cycle?
bool batch_stream_ok(mppi_handle ** hs, int n)
{
  mppi_handle * L = hs[0];
  for (int i = 0; i < n; ++i) {
    const mppi_handle * h = hs[i];
    if (!h->stream_layout || !h->params_in_arena || h->tail_mode != 0 || h->cfg.iteration_count != 1 || h->profiling ||
      h->cfg.regenerate_noises || h->nranks > 1)
    {
      L->err = std::string("batched launch not used: member ") + std::to_string(i) + " does not qualify this cycle";
      return false;
    }
  }
  return true;
}

// One cycle of the members [c0, c0 + n) of a stream-layout group (records built): ONE strided upload, then K2 / K3a /
// K3c / K4 launched once each with the robot as the last grid dimension; results as packets (tag) in each member's pinned
// result buffer.  first / last: the leader's events bracket the whole call.
mppi_status batch_stream_launch(mppi_handle * L, mppi_handle ** hs, int c0, int n, bool with_upload, uint32_t tag, bool first, bool last)
{
  unsigned inst = pick_stream_instance(stream_feature_need(hs[0]->last));
  size_t max_used = 0;
  for (int i = 0; i < n; ++i) {
    if (pick_stream_instance(stream_feature_need(hs[i]->last)) != inst) {inst = SF_ALL;}
    max_used = std::max(max_used, upload_bytes(hs[i]));
  }
  if (first && L->timing) {CUDA_TRY(L, cudaEventRecord(L->ev0, L->stream));}
  if (with_upload) {
    // the chunk's slices travel on the group's copy stream, i.e. beside the kernels of the previous chunk (the slices of
    // different chunks are disjoint; the previous STEP's kernels are done: its results have been delivered)
    const size_t off = L->arena_slice * static_cast<size_t>(c0);
    cudaEvent_t ev = L->ev_upload[(c0 / std::max(n, 1)) & 7];
    CUDA_TRY(L, cudaMemcpy2DAsync(L->arena_d + off, L->arena_slice, L->arena_h + off, L->arena_slice, max_used, n,
      cudaMemcpyHostToDevice, L->copy_stream));
    CUDA_TRY(L, cudaEventRecord(ev, L->copy_stream));
    CUDA_TRY(L, cudaStreamWaitEvent(L->stream, ev, 0));
  }
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    FusedJob & j = L->h_jobs[c0 + i];
    std::memset(&j, 0, sizeof(j));
    j.Pg = reinterpret_cast<const DevParams *>(h->d_params);
    j.cm = h->d_costmap;
    j.bufs = make_bufs(h, 0);
    j.B = h->B; j.T = h->T;
    j.host_res = h->h_res;
    h->wait_packets = true;
    h->zero_copy_now = false;
    h->ev_src = L;
    h->result_tag = tag;
    h->d2h_bytes = sizeof(uint2) * (3 * h->T + 2);
    h->h2d_bytes = with_upload ? upload_bytes(h) : 0;
  }
  const size_t off = sizeof(FusedJob) * static_cast<size_t>(c0), bytes = sizeof(FusedJob) * static_cast<size_t>(n);
  if (std::memcmp(L->jobs_sent.data() + off, L->h_jobs + c0, bytes) != 0) {
    CUDA_TRY(L, cudaMemcpyAsync(L->d_jobs + c0, L->h_jobs + c0, bytes, cudaMemcpyHostToDevice, L->stream));
    std::memcpy(L->jobs_sent.data() + off, L->h_jobs + c0, bytes);
  }
  const FusedJob * jobs = L->d_jobs + c0;
  const int T = L->T, B = L->B;
  {
    const int nthr = stream_block_threads(L);
    const int Tp = ((T + kStreamChunk - 1) / kStreamChunk) * kStreamChunk;
    const size_t smem = kHotBytes + sizeof(float) * 3 * (Tp + nthr);
    cudaError_t e;
    switch (inst) {
      case kSfOmniDefault: e = launch_stream_batch_instance<kSfOmniDefault, true>(L, jobs, n, nthr, smem); break;
      case kSfOmniDefaultFp: e = launch_stream_batch_instance<kSfOmniDefaultFp, true>(L, jobs, n, nthr, smem); break;
      case kSfObstaclesFp: e = launch_stream_batch_instance<kSfObstaclesFp, true>(L, jobs, n, nthr, smem); break;
      default: e = launch_stream_batch_instance<SF_ALL, false>(L, jobs, n, nthr, smem); break;
    }
    CUDA_TRY(L, e);
  }
  {
    const int grid = std::min((B + kUpdThreads - 1) / kUpdThreads, 148 * 8);
    path_costs_tm_batch_kernel<<<dim3(grid, n), kUpdThreads, k3_common_smem_bytes(), L->stream>>>(jobs);
    CUDA_TRY(L, cudaGetLastError());
  }
  const int chunks = (B + kWsChunk - 1) / kWsChunk;
  {
    const int gy = weighted_sums_row_groups(T, chunks * n);   // the rows are split less when many robots fill the machine
    weighted_sums_tm_batch_kernel<<<dim3(chunks, gy, n), kWsThreads, 0, L->stream>>>(jobs);
    CUDA_TRY(L, cudaGetLastError());
  }
  {
    const int merge_grid = (T + kMergeT - 1) / kMergeT;
    merge_finalize_batch_kernel<<<dim3(merge_grid, n), kUpdThreads, 0, L->stream>>>(jobs, chunks, 3 * T + 2, tag);
    CUDA_TRY(L, cudaGetLastError());
  }
  if (last && L->timing) {CUDA_TRY(L, cudaEventRecord(L->ev1, L->stream));}
  L->launches += 4;
  return MPPI_OK;
}

// The whole group, in chunks of kBatchChunk robots: records of a chunk are built (ins != nullptr) and the chunk is
// launched while the device still works on the previous ones.  Members of a chunk that does not qualify run one by one.
mppi_status batch_run_group(mppi_handle ** hs, const mppi_cycle_in * ins, mppi_cycle_out * outs, int n)
{
  mppi_handle * L = hs[0];
  CUDA_TRY(L, cudaSetDevice(L->device));
  mppi_status first = MPPI_OK;
  std::vector<char> pending(n, 0);
  if (L->batch_mode == 2) {
    // stream-layout group, in chunks: the records of a chunk are built, then the chunk is uploaded with one strided copy
    // and launched (four kernels) while the host builds the next chunk
    if (batch_stream_ok(hs, n)) {
      const uint32_t tag = 0x80000000u | (++L->batch_tag);   // never a tag of the fused kernel's epochs
      const int chunk = ins ? kStreamBatchChunk : n;
      for (int c0 = 0; c0 < n; c0 += chunk) {
        const int cn = std::min(chunk, n - c0);
        mppi_status s = MPPI_OK;
        for (int i = c0; i < c0 + cn && s == MPPI_OK; ++i) {
          if (ins) {
            s = build_params(hs[i], &ins[i], 0, kUnset, true);
            if (s == MPPI_OK) {s = stage_costmap(hs[i], ins[i].costmap);}
            if (s == MPPI_OK) {hs[i]->cycle_uploaded = true;}
          } else if (!hs[i]->cycle_uploaded) {
            s = fail(hs[i], MPPI_E_STATE, "mppi_optimize_batch_resident before mppi_upload_cycle");
          }
        }
        if (s == MPPI_OK) {s = batch_stream_launch(L, hs + c0, c0, cn, ins != nullptr, tag, c0 == 0, c0 + cn == n);}
        if (s == MPPI_OK) {
          for (int i = c0; i < c0 + cn; ++i) {pending[i] = 1;}
        } else if (first == MPPI_OK) {
          first = s;
        }
      }
      for (int i = 0; i < n; ++i) {
        if (!pending[i]) {continue;}
        const mppi_status f = finish_optimize(hs[i], outs ? &outs[i] : nullptr);
        if (f != MPPI_OK && first == MPPI_OK) {first = f;}
      }
      return first;
    }
    if (L->timing) {cudaEventRecord(L->ev0, L->stream);}
    for (int i = 0; i < n; ++i) {   // one by one on the shared stream
      mppi_status f = MPPI_OK;
      if (ins) {
        f = build_params(hs[i], &ins[i], 0, kUnset, true);
        if (f == MPPI_OK) {f = stage_costmap(hs[i], ins[i].costmap);}
        if (f == MPPI_OK) {hs[i]->cycle_uploaded = true;}
      } else if (!hs[i]->cycle_uploaded) {
        f = fail(hs[i], MPPI_E_STATE, "mppi_optimize_batch_resident before mppi_upload_cycle");
      }
      if (f == MPPI_OK) {f = enqueue_optimize(hs[i], ins != nullptr);}
      if (f == MPPI_OK) {f = finish_optimize(hs[i], outs ? &outs[i] : nullptr);}
      if (f != MPPI_OK && first == MPPI_OK) {first = f;}
    }
    return first;
  }
  // resident inputs: nothing to prepare on the host, one launch for the whole group
  const int chunk = ins ? kBatchChunk : n;
  for (int c0 = 0; c0 < n; c0 += chunk) {
    const int cn = std::min(chunk, n - c0);
    mppi_status s = MPPI_OK;
    for (int i = c0; i < c0 + cn && s == MPPI_OK; ++i) {
      if (ins) {
        s = build_params(hs[i], &ins[i], 0, kUnset, true);
        if (s == MPPI_OK) {s = stage_costmap(hs[i], ins[i].costmap);}
        if (s == MPPI_OK) {hs[i]->cycle_uploaded = true;}
      } else if (!hs[i]->cycle_uploaded) {
        s = fail(hs[i], MPPI_E_STATE, "mppi_optimize_batch_resident before mppi_upload_cycle");
      }
    }
    if (s == MPPI_OK) {s = batch_launch(L, hs + c0, c0, cn, ins != nullptr, c0 == 0, c0 + cn == n);}
    if (s == MPPI_OK) {
      for (int i = c0; i < c0 + cn; ++i) {pending[i] = 1;}
    } else if (s == MPPI_E_STATE) {
      // this chunk does not qualify: one by one on the shared stream (records are built already)
      if (c0 == 0 && L->timing) {cudaEventRecord(L->ev0, L->stream);}
      for (int i = c0; i < c0 + cn; ++i) {
        mppi_status f = hs[i]->cycle_uploaded ? enqueue_optimize(hs[i], ins != nullptr) : MPPI_E_STATE;
        if (f == MPPI_OK) {pending[i] = 1;} else if (first == MPPI_OK) {first = f;}
      }
      if (c0 + cn == n && L->timing) {cudaEventRecord(L->ev1, L->stream);}
    } else if (first == MPPI_OK) {
      first = s;
    }
  }
  for (int i = 0; i < n; ++i) {
    if (!pending[i]) {continue;}
    const mppi_status f = finish_optimize(hs[i], outs ? &outs[i] : nullptr);
    if (f != MPPI_OK && first == MPPI_OK) {first = f;}
  }
  return first;
}

}  // namespace

// =================================================================================================
extern "C" {

int32_t mppi_abi_version(void) {return MPPI_ABI_VERSION;}

#ifdef MPPI_TRACE
// tuning aid (only in -DMPPI_TRACE builds): copies the phase trace of the last kernels
int32_t mppi_debug_get_trace(long long * out, int32_t n)
{
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(out, mppi::g_trace, sizeof(long long) * std::min(n, 64)) == cudaSuccess ? 0 : 1;
}
#endif

void mppi_config_default(mppi_config * c)
{
  std::memset(c, 0, sizeof(*c));
  // Optimizer::getParams optimizer.cpp:69-84
  c->batch_size = 1000; c->time_steps = 56; c->iteration_count = 1;
  c->model_dt = 0.05f; c->temperature = 0.3f; c->gamma = 0.015f;
  c->vx_max = 0.5; c->vx_min = -0.35; c->vy_max = 0.5; c->wz_max = 1.9;
  c->vx_std = 0.2; c->vy_std = 0.2; c->wz_std = 0.4;
  c->motion_model = MPPI_MODEL_DIFF_DRIVE;
  c->ackermann_min_turning_r = 0.2;
}

void mppi_critic_default(int32_t kind, mppi_critic_desc * d)
{
  std::memset(d, 0, sizeof(*d));
  d->kind = kind; d->enabled = 1; d->cost_power = 1;
  d->trajectory_point_step = 4; d->max_path_occupancy_ratio = 0.07; d->use_path_orientations = 0;
  d->max_angle_to_furthest = 1.2; d->forward_preference = 1; d->consider_footprint = 0;
  d->near_goal_distance = 0.5; d->repulsion_weight = 1.5; d->critical_weight = 20.0;
  d->collision_margin_distance = 0.10; d->cost_scaling_factor = 10.0; d->inflation_radius = 0.55;
  d->critical_cost = 300.0;
  switch (kind) {
    case MPPI_CRITIC_CONSTRAINT: d->cost_weight = 4.0; break;                                      // constraint_critic.cpp:25-26
    case MPPI_CRITIC_COST: d->cost_weight = 3.81; d->collision_cost = 1000000.0; break;             // cost_critic.cpp:24-34
    case MPPI_CRITIC_GOAL: d->cost_weight = 5.0; d->threshold_to_consider = 1.4; break;             // goal_critic.cpp:27-29
    case MPPI_CRITIC_GOAL_ANGLE: d->cost_weight = 3.0; d->threshold_to_consider = 0.5; break;       // goal_angle_critic.cpp:24-27
    case MPPI_CRITIC_OBSTACLES: d->collision_cost = 10000.0; break;                                 // obstacles_critic.cpp:23-31
    case MPPI_CRITIC_PATH_ALIGN:
    case MPPI_CRITIC_PATH_ALIGN_LEGACY:                                                             // path_align_critic.cpp:29-38
      d->cost_weight = 10.0; d->threshold_to_consider = 0.5; d->offset_from_furthest = 20; break;
    case MPPI_CRITIC_PATH_ANGLE:                                                                    // path_angle_critic.cpp:35-46
      d->cost_weight = 2.0; d->threshold_to_consider = 0.5; d->offset_from_furthest = 4; break;
    case MPPI_CRITIC_PATH_FOLLOW:                                                                   // path_follow_critic.cpp:27-32
      d->cost_weight = 5.0; d->threshold_to_consider = 1.4; d->offset_from_furthest = 6; break;
    case MPPI_CRITIC_PREFER_FORWARD: d->cost_weight = 5.0; d->threshold_to_consider = 0.5; break;   // prefer_forward_critic.cpp:23-27
    case MPPI_CRITIC_TWIRLING: d->cost_weight = 10.0; break;                                        // twirling_critic.cpp:24-25
    case MPPI_CRITIC_VELOCITY_DEADBAND: d->cost_weight = 35.0; break;                               // velocity_deadband_critic.cpp:24-25
    default: break;
  }
}

const char * mppi_last_error(const mppi_handle * h) {return h ? h->err.c_str() : "null handle";}

void mppi_destroy(mppi_handle * h)
{
  if (!h) {return;}
  cudaSetDevice(h->device);
  if (h->stream) {cudaStreamSynchronize(h->stream);}
  if (h->batch_leader) {batch_unbind_group(h->batch_leader);}   // a group does not survive the loss of a member
  for (const auto & r : h->pinned_ranges) {cudaHostUnregister(const_cast<char *>(r.first));}
  drop_graphs(h);
  if (h->comm && g_nccl.CommDestroy) {g_nccl.CommDestroy(h->comm);}
  if (h->peer_mode) {
    for (int r = 0; r < h->nranks; ++r) {
      if (r != h->rank && h->peer_box[r]) {cudaIpcCloseMemHandle(h->peer_box[r]);}
    }
  }
  for (float * p : h->d_noise) {cudaFree(p);}
  for (float * p : h->d_samples) {cudaFree(p);}
  for (float * p : h->d_spill) {cudaFree(p);}
  for (float * p : h->d_inj) {cudaFree(p);}
  cudaFree(h->d_vis);
  cudaFree(h->d_vis);
  cudaFree(h->d_tmp); cudaFree(h->d_params); cudaFree(h->d_cs); cudaFree(h->d_crit_rows);
  cudaFree(h->d_end_xy); cudaFree(h->d_cells); cudaFree(h->d_costs); cudaFree(h->d_partials); cudaFree(h->d_ws_done); cudaFree(h->d_rank_partial);
  cudaFree(h->d_gathered); h->gathered_capacity = 0; cudaFree(h->d_out); cudaFree(h->d_st); cudaFree(h->d_hist); cudaFree(h->d_seq); cudaFree(h->d_epoch);
  if (h->ev_result) {cudaEventDestroy(h->ev_result);} cudaFree(h->d_mailbox);
  cudaFreeHost(h->h_params); cudaFreeHost(h->h_out); cudaFreeHost(h->h_res);
  cudaFree(h->d_pk); cudaFree(h->d_fepoch);
  if (h->ev0) {cudaEventDestroy(h->ev0);}
  if (h->ev1) {cudaEventDestroy(h->ev1);}
  for (auto & e : h->pev) {if (e) {cudaEventDestroy(e);}}
  if (h->stream) {cudaStreamDestroy(h->stream);}
  delete h;
}

mppi_status mppi_create(const mppi_config * cfg, mppi_handle ** out)
{
  if (!cfg || !out) {return MPPI_E_CONFIG;}
  *out = nullptr;
  mppi_handle * h = new mppi_handle();
  h->cfg = *cfg;
  *out = h;   // returned even on failure so that mppi_last_error() can be read; caller destroys it
  auto bad = [&](const char * m) {h->err = m; return MPPI_E_CONFIG;};
  if (cfg->batch_size < 1) {return bad("batch_size < 1");}
  if (cfg->time_steps < 2 || cfg->time_steps > MPPI_MAX_TIME_STEPS) {return bad("time_steps must be in [2, MPPI_MAX_TIME_STEPS]");}
  if (cfg->iteration_count < 1) {return bad("iteration_count < 1");}
  if (cfg->motion_model < MPPI_MODEL_DIFF_DRIVE || cfg->motion_model > MPPI_MODEL_ACKERMANN) {
    return bad("Model is not valid! Valid options are DiffDrive, Omni, or Ackermann");   // optimizer.cpp:421-424
  }
  if (!(cfg->temperature > 0.0f) || !(cfg->model_dt > 0.0f)) {return bad("temperature and model_dt must be > 0");}
  if (!(cfg->vx_std > 0.0f) || !(cfg->vy_std > 0.0f) || !(cfg->wz_std > 0.0f)) {return bad("sampling std must be > 0");}
  h->B = cfg->batch_size; h->T = cfg->time_steps; h->device = cfg->device;
  h->base = {cfg->vx_max, cfg->vx_min, cfg->vy_max, cfg->wz_max};
  h->cur = h->base;
  std::memset(&h->robot, 0, sizeof(h->robot));
  if (const char * e = std::getenv("MPPI_SEGMENTS")) {h->segments_override = std::atoi(e);}
  if (const char * e = std::getenv("MPPI_STREAM_THREADS")) {
    h->stream_threads_override = std::max(32, std::min(kStreamThreads, (std::atoi(e) / 32) * 32));
  }
  if (const char * e = std::getenv("MPPI_NO_GRAPH")) {h->use_graph = std::atoi(e) == 0;}
  if (const char * e = std::getenv("MPPI_FUSED")) {h->fused_enabled = std::atoi(e) != 0;}
  if (const char * e = std::getenv("MPPI_ZERO_COPY")) {h->zero_copy_enabled = std::atoi(e) != 0;}
  if (const char * e = std::getenv("MPPI_COOP")) {h->coop_launch = std::atoi(e) != 0;}
  if (const char * e = std::getenv("MPPI_STREAM_PACKETS")) {h->packets_enabled = std::atoi(e) != 0;}
  if (const char * e = std::getenv("MPPI_PDL")) {h->pdl_enabled = std::atoi(e) != 0;}
  if (const char * e = std::getenv("MPPI_SCAN")) {h->scan_mode = std::strcmp(e, "warp") == 0 ? 1 : 0;}
  if (const char * e = std::getenv("MPPI_WS_TMA")) {h->ws_tma_enabled = std::atoi(e) != 0;}
  {
    // batches too small to fill the GPU with one thread per trajectory keep the latency-oriented tile kernel
    long long stream_min = 8192;    // measured cross-over on B200 (profiles/): below it the tile kernel wins
    if (const char * e = std::getenv("MPPI_STREAM_MIN_BATCH")) {stream_min = std::atoll(e);}
    h->stream_layout = cfg->batch_size >= stream_min;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    h->err = "no CUDA device: this library has no CPU fallback";
    return MPPI_E_CUDA;
  }
  CUDA_TRY(h, cudaSetDevice(h->device));
  {
    const int big = 227 * 1024;
    CUDA_TRY(h, cudaFuncSetAttribute(rollout_score_kernel<SF_ALL, false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(rollout_score_kernel<SF_ALL, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(rollout_score_kernel<SF_ALL, false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(rollout_score_kernel<kSfOmniDefault, true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(rollout_score_kernel<kSfOmniDefaultFp, true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(rollout_score_kernel<kSfObstaclesFp, true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  }
  {
    const int big = kFusedSmemMax;   // the kernel also has a little static shared memory
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_kernel<SF_ALL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_kernel<kSfOmniDefault, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_kernel<kSfOmniDefaultFp, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_kernel<kSfObstaclesFp, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_batch_kernel<SF_ALL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_batch_kernel<kSfOmniDefault, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_batch_kernel<kSfOmniDefaultFp, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CUDA_TRY(h, cudaFuncSetAttribute(tile_fused_batch_kernel<kSfObstaclesFp, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    int coop = 0;
    CUDA_TRY(h, cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->device));
    CUDA_TRY(h, cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device));
    if (!coop) {h->fused_enabled = false;}
  }
  CUDA_TRY(h, cudaFuncSetAttribute(path_softmax_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
    static_cast<int>(k3_tile_smem_bytes(MPPI_MAX_TIME_STEPS))));
  CUDA_TRY(h, cudaFuncSetAttribute(weighted_sums_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
    static_cast<int>(ps_smem_bytes())));
  CUDA_TRY(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CUDA_TRY(h, cudaEventCreate(&h->ev0));
  CUDA_TRY(h, cudaEventCreate(&h->ev1));
  for (auto & e : h->pev) {CUDA_TRY(h, cudaEventCreate(&e));}
  const size_t B = h->B, T = h->T, plane = B * T * sizeof(float);
  // kNoisePadRows zeroed rows behind every noise plane: the stream kernel prefetches past the horizon without a clamp
  const size_t noise_plane = plane + static_cast<size_t>(kNoisePadRows) * B * sizeof(float);
  if (h->stream_layout && (T + kNoisePadRows) * B >= (1ull << 32)) {
    return bad("batch_size * time_steps too large for the 32-bit offsets of the stream layout");
  }
  for (int i = 0; i < 3; ++i) {
    CUDA_TRY(h, cudaMalloc(&h->d_noise[i], noise_plane));
    CUDA_TRY(h, cudaMalloc(&h->d_samples[i], plane));
    CUDA_TRY(h, cudaMalloc(&h->d_spill[i], plane));
    CUDA_TRY(h, cudaMemsetAsync(h->d_noise[i], 0, noise_plane, h->stream));
  }
  if (h->stream_layout && h->ws_tma_enabled) {h->ws_tma_ok = make_noise_maps(h);}
  CUDA_TRY(h, cudaMalloc(&h->d_cells, B * T * sizeof(int)));
  CUDA_TRY(h, cudaMalloc(&h->d_params, kParamsCapacity + 256));
  CUDA_TRY(h, cudaMalloc(&h->d_cs, 3 * T * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d_crit_rows, (kMaxCritics + kGammaRows) * B * sizeof(float)));
  CUDA_TRY(h, cudaMemsetAsync(h->d_crit_rows, 0, (kMaxCritics + kGammaRows) * B * sizeof(float), h->stream));
  CUDA_TRY(h, cudaMalloc(&h->d_end_xy, 2 * B * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d_costs, B * sizeof(float)));
  h->upd_blocks = static_cast<int>((B + kUpdRows - 1) / kUpdRows);
  const size_t stride = 3 * T + 2;
  CUDA_TRY(h, cudaMalloc(&h->d_partials, h->upd_blocks * stride * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d_rank_partial, stride * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d_ws_done, kWsDoneSlots * sizeof(unsigned)));
  CUDA_TRY(h, cudaMemsetAsync(h->d_ws_done, 0, kWsDoneSlots * sizeof(unsigned), h->stream));
  CUDA_TRY(h, cudaMalloc(&h->d_out, (stride + 8) * sizeof(float)));
  CUDA_TRY(h, cudaMemsetAsync(h->d_out, 0, (stride + 8) * sizeof(float), h->stream));
  CUDA_TRY(h, cudaMalloc(&h->d_hist, 12 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d_epoch, sizeof(unsigned long long)));
  CUDA_TRY(h, cudaEventCreate(&h->ev_result));
  CUDA_TRY(h, cudaMalloc(&h->d_seq, sizeof(unsigned)));
  CUDA_TRY(h, cudaMemsetAsync(h->d_seq, 0, sizeof(unsigned), h->stream));
  CUDA_TRY(h, cudaMalloc(&h->d_st, sizeof(DevState)));
  if (!h->stream_layout) {
    const size_t n_pk = static_cast<size_t>(h->upd_blocks) * (2 + stride) + stride;
    CUDA_TRY(h, cudaMalloc(&h->d_pk, n_pk * sizeof(uint2)));
    CUDA_TRY(h, cudaMemsetAsync(h->d_pk, 0, n_pk * sizeof(uint2), h->stream));
  }
  CUDA_TRY(h, cudaMalloc(&h->d_fepoch, sizeof(unsigned)));
  CUDA_TRY(h, cudaMemsetAsync(h->d_fepoch, 0, sizeof(unsigned), h->stream));
  CUDA_TRY(h, cudaHostAlloc(&h->h_res, (stride + 8) * sizeof(uint2), cudaHostAllocMapped | cudaHostAllocPortable));
  std::memset(h->h_res, 0, (stride + 8) * sizeof(uint2));
  CUDA_TRY(h, cudaHostAlloc(&h->h_params, kParamsCapacity + 256, cudaHostAllocMapped | cudaHostAllocPortable));
  CUDA_TRY(h, cudaMallocHost(&h->h_out, (stride + 8) * sizeof(float)));
  return do_reset(h);
}

mppi_status mppi_reset(mppi_handle * h)
{
  if (!h) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  return do_reset(h);
}

mppi_status mppi_set_critics(mppi_handle * h, const mppi_critic_desc * critics, int32_t n)
{
  if (!h || n < 0 || (n > 0 && !critics)) {return MPPI_E_CONFIG;}
  if (n > MPPI_MAX_CRITICS) {return fail(h, MPPI_E_CONFIG, "too many critics");}
  bool seen[MPPI_CRITIC_KIND_COUNT] = {};
  for (int i = 0; i < n; ++i) {
    const int k = critics[i].kind;
    if (k < 0 || k >= MPPI_CRITIC_KIND_COUNT) {return fail(h, MPPI_E_CONFIG, "unknown critic kind");}
    if (seen[k]) {return fail(h, MPPI_E_CONFIG, "a critic kind may appear only once in the critics list");}
    seen[k] = true;
  }
  h->critics.assign(critics, critics + n);
  h->cycle_uploaded = false;
  return MPPI_OK;
}

mppi_status mppi_set_robot(mppi_handle * h, const mppi_robot_desc * robot)
{
  if (!h || !robot) {return MPPI_E_CONFIG;}
  if (robot->footprint_size < 0 || robot->footprint_size > MPPI_MAX_FOOTPRINT) {return fail(h, MPPI_E_CONFIG, "footprint_size out of range");}
  h->robot = *robot;
  h->cycle_uploaded = false;
  return MPPI_OK;
}

mppi_status mppi_set_speed_limit(mppi_handle * h, double speed_limit, int32_t percentage)
{
  if (!h) {return MPPI_E_CONFIG;}
  Constraints & s = h->cur;
  const Constraints & b = h->base;
  if (speed_limit == 0.0) {        // nav2_costmap_2d::NO_SPEED_LIMIT
    s = b;
  } else {
    const double ratio = percentage ? speed_limit / 100.0 : speed_limit / b.vx_max;
    s.vx_max = b.vx_max * ratio; s.vx_min = b.vx_min * ratio; s.vy = b.vy * ratio; s.wz = b.wz * ratio;
  }
  h->cycle_uploaded = false;
  return MPPI_OK;
}

mppi_status mppi_get_constraints(const mppi_handle * h, float out4[4])
{
  if (!h || !out4) {return MPPI_E_CONFIG;}
  out4[0] = h->cur.vx_max; out4[1] = h->cur.vx_min; out4[2] = h->cur.vy; out4[3] = h->cur.wz;
  return MPPI_OK;
}

mppi_status mppi_set_noise(mppi_handle * h, const float * vx, const float * vy, const float * wz)
{
  if (!h || !vx || !wz) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  const size_t plane = static_cast<size_t>(h->B) * h->T * sizeof(float);
  const float * src[3] = {vx, vy, wz};
  if (h->stream_layout) {
    mppi_status s = ensure_tmp(h);
    if (s != MPPI_OK) {return s;}
  }
  for (int i = 0; i < 3; ++i) {
    if (!src[i]) {
      CUDA_TRY(h, cudaMemsetAsync(h->d_noise[i], 0, plane, h->stream));
      continue;
    }
    if (!h->stream_layout) {
      CUDA_TRY(h, cudaMemcpyAsync(h->d_noise[i], src[i], plane, cudaMemcpyHostToDevice, h->stream));
    } else {
      // caller's layout is [B][T]; the stream layout keeps [T][B]
      CUDA_TRY(h, cudaMemcpyAsync(h->d_tmp, src[i], plane, cudaMemcpyHostToDevice, h->stream));
      const dim3 grid((h->T + 31) / 32, (h->B + 31) / 32), block(32, 8);
      transpose_tb_to_bt_kernel<float><<<grid, block, 0, h->stream>>>(h->d_tmp, h->d_noise[i], h->B, h->T);
      CUDA_TRY(h, cudaGetLastError());
    }
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_generate_noise(mppi_handle * h, uint64_t stream)
{
  if (!h) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  const long long total = static_cast<long long>(h->B) * ((h->T + 3) / 4);
  const int blocks = static_cast<int>(std::min<long long>((total + 255) / 256, 148LL * 16));
  noise_philox_kernel<<<std::max(blocks, 1), 256, 0, h->stream>>>(
    h->d_noise[0], h->d_noise[1], h->d_noise[2], h->B, h->T, h->cfg.vx_std, h->cfg.vy_std, h->cfg.wz_std,
    holonomic(h) ? 1 : 0, h->cfg.seed, stream, static_cast<uint64_t>(h->cfg.shard_offset), h->stream_layout ? 1 : 0, nullptr);
  CUDA_TRY(h, cudaGetLastError());
  h->launches++;
  h->noise_stream = stream + 1;   // a later reset() draws the next stream
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return sync_epoch(h);
}

mppi_status mppi_get_noise(mppi_handle * h, float * vx, float * vy, float * wz)
{
  if (!h || !vx || !vy || !wz) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  const size_t plane = static_cast<size_t>(h->B) * h->T * sizeof(float);
  float * dst[3] = {vx, vy, wz};
  for (int i = 0; i < 3; ++i) {
    if (h->stream_layout) {
      const mppi_status s = fetch_time_major<float>(h, h->d_noise[i], dst[i]);
      if (s != MPPI_OK) {return s;}
    } else {
      CUDA_TRY(h, cudaMemcpyAsync(dst[i], h->d_noise[i], plane, cudaMemcpyDeviceToHost, h->stream));
    }
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_set_control_sequence(mppi_handle * h, const float * vx, const float * vy, const float * wz)
{
  if (!h || !vx || !vy || !wz) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  const size_t n = h->T * sizeof(float);
  CUDA_TRY(h, cudaMemcpyAsync(h->d_cs, vx, n, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_cs + h->T, vy, n, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_cs + 2 * h->T, wz, n, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_get_control_sequence(mppi_handle * h, float * vx, float * vy, float * wz)
{
  if (!h || !vx || !vy || !wz) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  const size_t n = h->T * sizeof(float);
  CUDA_TRY(h, cudaMemcpyAsync(vx, h->d_cs, n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(vy, h->d_cs + h->T, n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(wz, h->d_cs + 2 * h->T, n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_shift_control_sequence(mppi_handle * h)
{
  if (!h) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  shift_control_sequence_kernel<<<1, 256, 0, h->stream>>>(h->d_cs, h->T, holonomic(h) ? 1 : 0);
  CUDA_TRY(h, cudaGetLastError());
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_set_outputs(mppi_handle * h, uint32_t want_mask)
{
  if (!h) {return MPPI_E_CONFIG;}
  h->want_mask = want_mask;
  h->cycle_uploaded = false;
  return MPPI_OK;
}

mppi_status mppi_upload_cycle(mppi_handle * h, const mppi_cycle_in * in)
{
  if (!h || !in) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s = build_params(h, in, 0, kUnset, true);
  if (s != MPPI_OK) {return s;}
  if ((s = stage_costmap(h, in->costmap)) != MPPI_OK) {return s;}
  if ((s = enqueue_uploads(h)) != MPPI_OK) {return s;}
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->cycle_uploaded = true;
  return MPPI_OK;
}

mppi_status mppi_optimize_resident(mppi_handle * h, mppi_cycle_out * out)
{
  if (!h) {return MPPI_E_CONFIG;}
  if (!h->cycle_uploaded) {return fail(h, MPPI_E_STATE, "mppi_optimize_resident before mppi_upload_cycle");}
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s = enqueue_optimize(h, false);
  if (s != MPPI_OK) {return s;}
  return finish_optimize(h, out);
}

// prepare() + optimize(): pack the cycle record, stage the costmap, then ONE graph launch does
// H2D(record) + H2D(costmap) + K2 + K3 + D2H(result); the call returns after the result is in host memory
static mppi_status optimize_begin(mppi_handle * h, const mppi_cycle_in * in)
{
  if (!h || !in) {return MPPI_E_CONFIG;}
  const uint64_t t_a = now_ns();
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s = build_params(h, in, 0, kUnset, true);
  if (s != MPPI_OK) {return s;}
  const uint64_t t_b = now_ns();
  if ((s = stage_costmap(h, in->costmap)) != MPPI_OK) {return s;}
  h->host_ns[0] += t_b - t_a;
  h->host_ns[1] += now_ns() - t_b;
  h->cycle_uploaded = true;
  return enqueue_optimize(h, true);
}

mppi_status mppi_optimize(mppi_handle * h, const mppi_cycle_in * in, mppi_cycle_out * out)
{
  mppi_status s = optimize_begin(h, in);
  if (s != MPPI_OK) {return s;}
  return finish_optimize(h, out);
}

// Optimizer::evalControl (optimizer.cpp:134-155) without the fallback loop: prepare + optimize, and, when the
// optimisation did not fail, savitskyGolayFilter + getControlFromSequenceAsTwist + shiftControlSequence on the device.
mppi_status mppi_eval_control(mppi_handle * h, const mppi_cycle_in * in, int32_t shift_control_sequence, mppi_cycle_out * out, float cmd_out[3])
{
  if (!h || !in) {return MPPI_E_CONFIG;}
  if (h->nranks > 1 && !h->peer_mode) {return fail(h, MPPI_E_STATE, "mppi_eval_control on an NCCL-sharded handle: use mppi_optimize + the host tail");}
  h->tail_mode = shift_control_sequence ? 2 : 1;
  mppi_status s = optimize_begin(h, in);
  if (s == MPPI_OK) {s = finish_optimize(h, out);}
  h->tail_mode = 0;
  if (s != MPPI_OK) {return s;}
  if (cmd_out) {std::memcpy(cmd_out, h->h_out + 3 * h->T + 2, 3 * sizeof(float));}
  return MPPI_OK;
}

mppi_status mppi_set_control_history(mppi_handle * h, const float hist12[12])
{
  if (!h || !hist12) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_hist, hist12, 12 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_get_control_history(mppi_handle * h, float hist12[12])
{
  if (!h || !hist12) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaMemcpyAsync(hist12, h->d_hist, 12 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

// Multi-robot server: bind n handles of one device (same batch_size / time_steps, tile layout, not sharded) into a
// group.  They share the first handle's stream from here on, and mppi_optimize_batch[_resident] over exactly this group
// (same order) becomes ONE kernel launch for all robots.  Everything else keeps working on bound handles.
mppi_status mppi_batch_bind(mppi_handle ** hs, int32_t n)
{
  if (!hs || n < 1 || !hs[0]) {return MPPI_E_CONFIG;}
  mppi_handle * L = hs[0];
  // mode 2 (default): the members move to the stream layout and the group runs as four batched kernels; mode 1
  // (MPPI_BATCH_MODE=tile): the members stay in the tile layout, one ticketed fused kernel per 16 robots
  int mode = 2;
  if (const char * e = std::getenv("MPPI_BATCH_MODE")) {mode = std::strcmp(e, "tile") == 0 ? 1 : 2;}
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    if (!h) {return MPPI_E_CONFIG;}
    if (h->device != L->device || h->B != L->B || h->T != L->T) {return fail(L, MPPI_E_CONFIG, "mppi_batch_bind: handles must share device, batch_size and time_steps");}
    if ((mode == 1 && h->stream_layout) || h->nranks > 1 || h->cfg.regenerate_noises) {return fail(L, MPPI_E_CONFIG, "mppi_batch_bind: unsharded handles without regenerate_noises only (tile mode: tile layout only)");}
    for (int k = 0; k < i; ++k) {if (hs[k] == h) {return fail(L, MPPI_E_CONFIG, "mppi_batch_bind: duplicate handle");}}
  }
  for (int i = 0; i < n; ++i) {
    if (hs[i]->batch_leader) {batch_unbind_group(hs[i]->batch_leader);}
  }
  CUDA_TRY(L, cudaSetDevice(L->device));
  CUDA_TRY(L, cudaHostAlloc(&L->h_jobs, sizeof(FusedJob) * static_cast<size_t>(n), cudaHostAllocDefault));
  CUDA_TRY(L, cudaMalloc(&L->d_jobs, sizeof(FusedJob) * static_cast<size_t>(n)));
  CUDA_TRY(L, cudaMalloc(&L->d_ticket, sizeof(unsigned)));
  CUDA_TRY(L, cudaMemsetAsync(L->d_ticket, 0, sizeof(unsigned), L->stream));
  L->ticket_base = 0;
  L->jobs_sent.assign(sizeof(FusedJob) * static_cast<size_t>(n), 0);
  std::memset(L->h_jobs, 0, sizeof(FusedJob) * static_cast<size_t>(n));
  L->batch_group.assign(hs, hs + n);
  L->batch_mode = mode;
  L->batch_tag = 0;
  if (mode == 2) {
    size_t cap = 64 * 1024;
    for (int i = 0; i < n; ++i) {cap = std::max(cap, hs[i]->costmap_capacity);}
    L->arena_slice = (kParamsCapacity + 256 + cap + 255) & ~static_cast<size_t>(255);
    CUDA_TRY(L, cudaHostAlloc(&L->arena_h, L->arena_slice * n, cudaHostAllocMapped | cudaHostAllocPortable));
    CUDA_TRY(L, cudaMalloc(&L->arena_d, L->arena_slice * n));
    CUDA_TRY(L, cudaStreamCreateWithFlags(&L->copy_stream, cudaStreamNonBlocking));
    for (auto & e : L->ev_upload) {CUDA_TRY(L, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));}
  }
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    drop_graphs(h);
    if (mode == 2) {
      const mppi_status s = to_stream_layout(h);
      if (s != MPPI_OK) {batch_unbind_group(L); return s;}
      cudaFreeHost(h->h_params); cudaFree(h->d_params);
      h->h_params = L->arena_h + L->arena_slice * i;
      h->d_params = L->arena_d + L->arena_slice * i;
      h->h_costmap = nullptr; h->d_costmap = nullptr;
      h->costmap_capacity = L->arena_slice - kParamsCapacity - 256;
      h->params_in_arena = true;
      h->cycle_uploaded = false;
      std::memset(h->h_res, 0, (3 * static_cast<size_t>(h->T) + 10) * sizeof(uint2));
    }
    h->batch_leader = L;
    if (h != L) {h->own_stream = h->stream; h->stream = L->stream;}
  }
  return MPPI_OK;
}

mppi_status mppi_batch_unbind(mppi_handle * any_member)
{
  if (!any_member) {return MPPI_E_CONFIG;}
  batch_unbind_group(any_member->batch_leader);
  return MPPI_OK;
}

mppi_status mppi_optimize_batch(mppi_handle ** hs, const mppi_cycle_in * ins, mppi_cycle_out * outs, int32_t n)
{
  if (!hs || !ins || n < 0) {return MPPI_E_CONFIG;}
  if (batch_is_group(hs, n)) {return batch_run_group(hs, ins, outs, n);}
  mppi_status first = MPPI_OK;
  std::vector<char> launched(n, 0);
  for (int i = 0; i < n; ++i) {
    const mppi_status s = optimize_begin(hs[i], &ins[i]);
    launched[i] = s == MPPI_OK;
    if (s != MPPI_OK && first == MPPI_OK) {first = s;}
  }
  for (int i = 0; i < n; ++i) {
    if (!launched[i]) {continue;}
    cudaSetDevice(hs[i]->device);
    const mppi_status s = finish_optimize(hs[i], outs ? &outs[i] : nullptr);
    if (s != MPPI_OK && first == MPPI_OK) {first = s;}
  }
  return first;
}

// the same over inputs that are already resident (mppi_upload_cycle on every handle): the measurement leg of the
// multi-robot workload
mppi_status mppi_optimize_batch_resident(mppi_handle ** hs, mppi_cycle_out * outs, int32_t n)
{
  if (!hs || n < 0) {return MPPI_E_CONFIG;}
  if (batch_is_group(hs, n)) {return batch_run_group(hs, nullptr, outs, n);}
  mppi_status first = MPPI_OK;
  std::vector<char> launched(n, 0);
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = hs[i];
    mppi_status s = MPPI_OK;
    if (!h) {
      s = MPPI_E_CONFIG;
    } else if (!h->cycle_uploaded) {
      s = fail(h, MPPI_E_STATE, "mppi_optimize_batch_resident before mppi_upload_cycle");
    } else if (cudaSetDevice(h->device) != cudaSuccess) {
      s = fail(h, MPPI_E_CUDA, "cudaSetDevice");
    } else {
      s = enqueue_optimize(h, false);
    }
    launched[i] = s == MPPI_OK;
    if (s != MPPI_OK && first == MPPI_OK) {first = s;}
  }
  for (int i = 0; i < n; ++i) {
    if (!launched[i]) {continue;}
    cudaSetDevice(hs[i]->device);
    const mppi_status s = finish_optimize(hs[i], outs ? &outs[i] : nullptr);
    if (s != MPPI_OK && first == MPPI_OK) {first = s;}
  }
  return first;
}

// device time of the last batch call over these handles (same device, timing on): from the first handle's start event
// to the latest end event.  The handles run on their own streams, so the per-handle device_ms overlap.
mppi_status mppi_batch_span_ms(mppi_handle ** hs, int32_t n, float * ms_out)
{
  if (!hs || n < 1 || !ms_out || !hs[0]) {return MPPI_E_CONFIG;}
  float span = 0.0f;
  for (int i = 0; i < n; ++i) {
    if (!hs[i] || !hs[i]->timing) {return MPPI_E_STATE;}
    float ms = 0.0f;
    const mppi_handle * e0 = hs[0]->ev_src ? hs[0]->ev_src : hs[0];
    const mppi_handle * e1 = hs[i]->ev_src ? hs[i]->ev_src : hs[i];
    if (cudaEventElapsedTime(&ms, e0->ev0, e1->ev1) != cudaSuccess) {
      cudaGetLastError();
      return fail(hs[i], MPPI_E_STATE, "mppi_batch_span_ms: no completed batch call to read");
    }
    span = std::max(span, ms);
  }
  *ms_out = span;
  return MPPI_OK;
}

mppi_status mppi_get_trajectories(mppi_handle * h, float * x, float * y, float * yaw)
{
  if (!h || !x || !y || !yaw) {return MPPI_E_CONFIG;}
  if (!h->spilled_traj) {return fail(h, MPPI_E_STATE, "trajectories were not materialised: mppi_set_outputs(MPPI_WANT_TRAJECTORIES) before optimize");}
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s;
  if ((s = fetch_time_major<float>(h, h->d_spill[0], x)) != MPPI_OK) {return s;}
  if ((s = fetch_time_major<float>(h, h->d_spill[1], y)) != MPPI_OK) {return s;}
  return fetch_time_major<float>(h, h->d_spill[2], yaw);
}

// The TrajectoryVisualizer (trajectory_visualizer.cpp:86-108) draws every trajectory_step-th candidate at every
// time_step-th step: materialise exactly that lattice in K2 (a few percent of the traffic of the full planes).
mppi_status mppi_set_visualization(mppi_handle * h, int32_t trajectory_step, int32_t time_step)
{
  if (!h || trajectory_step < 0 || time_step < 0 || (trajectory_step == 0) != (time_step == 0)) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  drop_graphs(h);
  h->vis_b_step = trajectory_step; h->vis_t_step = time_step; h->vis_valid = false;
  if (trajectory_step > 0) {
    const size_t nb = (h->B + trajectory_step - 1) / trajectory_step, nt = (h->T + time_step - 1) / time_step;
    if (2 * nb * nt > h->vis_capacity) {
      cudaFree(h->d_vis);
      h->d_vis = nullptr; h->vis_capacity = 0;
      CUDA_TRY(h, cudaMalloc(&h->d_vis, 2 * nb * nt * sizeof(float)));
      h->vis_capacity = 2 * nb * nt;
    }
  }
  return MPPI_OK;
}

// x, y: [ceil(B / trajectory_step)][ceil(T / time_step)] row-major = trajectories.x(i * trajectory_step, j * time_step)
mppi_status mppi_get_visualization(mppi_handle * h, float * x, float * y)
{
  if (!h || !x || !y) {return MPPI_E_CONFIG;}
  if (!h->vis_valid) {return fail(h, MPPI_E_STATE, "mppi_set_visualization before optimize");}
  CUDA_TRY(h, cudaSetDevice(h->device));
  const int nb = (h->B + h->vis_b_step - 1) / h->vis_b_step, nt = (h->T + h->vis_t_step - 1) / h->vis_t_step;
  mppi_status s = ensure_tmp(h);
  if (s != MPPI_OK) {return s;}
  const dim3 grid((nb + 31) / 32, (nt + 31) / 32), block(32, 8);
  float * dst[2] = {x, y};
  for (int k = 0; k < 2; ++k) {
    transpose_tb_to_bt_kernel<float><<<grid, block, 0, h->stream>>>(h->d_vis + static_cast<size_t>(k) * nt * nb, h->d_tmp, nt, nb);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(dst[k], h->d_tmp, static_cast<size_t>(nb) * nt * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  }
  return MPPI_OK;
}

mppi_status mppi_get_cells(mppi_handle * h, int32_t * cells)
{
  if (!h || !cells) {return MPPI_E_CONFIG;}
  if (!h->spilled_cells) {return fail(h, MPPI_E_STATE, "cell indices were not materialised: mppi_set_outputs(MPPI_WANT_CELLS) before optimize");}
  CUDA_TRY(h, cudaSetDevice(h->device));
  return fetch_time_major<int>(h, h->d_cells, cells);
}

mppi_status mppi_get_costs(mppi_handle * h, float * costs)
{
  if (!h || !costs) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaMemcpyAsync(costs, h->d_costs, h->B * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_get_critic_costs(mppi_handle * h, int32_t index, float * costs)
{
  if (!h || !costs) {return MPPI_E_CONFIG;}
  if (!h->have_rows) {return fail(h, MPPI_E_STATE, "no optimize has run yet");}
  if (!h->last.want_critic_rows) {return fail(h, MPPI_E_STATE, "request the rows first: mppi_set_outputs(MPPI_WANT_CRITIC_COSTS)");}
  if (index < 0 || index >= static_cast<int>(h->critics.size())) {return fail(h, MPPI_E_CONFIG, "critic index out of range");}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaMemcpyAsync(costs, h->d_crit_rows + static_cast<size_t>(index) * h->B, h->B * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_get_optimized_trajectory(mppi_handle * h, double pose_x, double pose_y, double pose_yaw, float * traj_t3)
{
  if (!h || !traj_t3) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s = ensure_tmp(h);
  if (s != MPPI_OK) {return s;}
  optimized_trajectory_kernel<<<1, 32, 0, h->stream>>>(h->d_cs, h->d_tmp, h->T, holonomic(h) ? 1 : 0, h->cfg.model_dt, pose_x, pose_y,
    static_cast<float>(pose_yaw));
  CUDA_TRY(h, cudaGetLastError());
  CUDA_TRY(h, cudaMemcpyAsync(traj_t3, h->d_tmp, 3 * h->T * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return MPPI_OK;
}

mppi_status mppi_integrate_state_velocities(
  mppi_handle * h, double pose_x, double pose_y, double pose_yaw, const float * vx, const float * vy, const float * wz,
  float * x, float * y, float * yaw)
{
  if (!h || !vx || !vy || !wz || !x || !y || !yaw) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s = ensure_injection_buffers(h);
  if (s != MPPI_OK) {return s;}
  const size_t plane = static_cast<size_t>(h->B) * h->T * sizeof(float);
  CUDA_TRY(h, cudaMemcpyAsync(h->d_inj[0], vx, plane, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_inj[1], vy, plane, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_inj[2], wz, plane, cudaMemcpyHostToDevice, h->stream));
  // a one-point dummy path and a 1x1 map: no critic runs in this mode
  static const float zero = 0.0f;
  static const uint8_t cell = 0;
  mppi_cycle_in in;
  std::memset(&in, 0, sizeof(in));
  in.pose_x = pose_x; in.pose_y = pose_y; in.pose_yaw = pose_yaw;
  in.goal_checker_xy_tolerance = -1.0;
  in.path_size = 1; in.path_x = &zero; in.path_y = &zero; in.path_yaw = &zero;
  in.costmap.cells = &cell; in.costmap.size_x = 1; in.costmap.size_y = 1; in.costmap.resolution = 1.0;
  const uint32_t keep_mask = h->want_mask;
  h->want_mask = 0;
  s = build_params(h, &in, 1, kUnset, false);
  h->want_mask = keep_mask;
  if (s != MPPI_OK) {return s;}
  if ((s = stage_costmap(h, in.costmap)) != MPPI_OK) {return s;}
  if ((s = enqueue_uploads(h)) != MPPI_OK) {return s;}
  h->cycle_uploaded = false;
  if ((s = launch_rollout(h, 1)) != MPPI_OK) {return s;}
  // K2 raised nothing persistent except the exchange-1 words; clear them for the next optimize
  CUDA_TRY(h, cudaMemsetAsync(h->d_st, 0, sizeof(DevState), h->stream));
  if ((s = fetch_time_major<float>(h, h->d_spill[0], x)) != MPPI_OK) {return s;}
  if ((s = fetch_time_major<float>(h, h->d_spill[1], y)) != MPPI_OK) {return s;}
  return fetch_time_major<float>(h, h->d_spill[2], yaw);
}

mppi_status mppi_score_trajectories(
  mppi_handle * h, const mppi_cycle_in * in, const float * vx, const float * vy, const float * wz, const float * x,
  const float * y, const float * yaw, float * costs_inout, uint32_t * furthest_inout, int32_t * fail_flag_out)
{
  if (!h || !in || !vx || !vy || !wz || !x || !y || !yaw || !costs_inout) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  mppi_status s = ensure_injection_buffers(h);
  if (s != MPPI_OK) {return s;}
  const size_t plane = static_cast<size_t>(h->B) * h->T * sizeof(float);
  const float * src[6] = {vx, vy, wz, x, y, yaw};
  for (int i = 0; i < 6; ++i) {
    CUDA_TRY(h, cudaMemcpyAsync(h->d_inj[i], src[i], plane, cudaMemcpyHostToDevice, h->stream));
  }
  CUDA_TRY(h, cudaMemcpyAsync(h->d_costs, costs_inout, h->B * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  const unsigned preset = furthest_inout ? *furthest_inout : kUnset;
  const float first_pose[2] = {x[0], y[0]};   // trajectories(0, 0): utils::findPathTrajectoryInitialPoint
  s = build_params(h, in, 2, preset, true, first_pose);
  if (s != MPPI_OK) {return s;}
  if ((s = stage_costmap(h, in->costmap)) != MPPI_OK) {return s;}
  if ((s = enqueue_uploads(h)) != MPPI_OK) {return s;}
  h->cycle_uploaded = false;
  if ((s = launch_rollout(h, 2)) != MPPI_OK) {return s;}
  if ((s = launch_update(h, 2, 0)) != MPPI_OK) {return s;}
  CUDA_TRY(h, cudaMemcpyAsync(h->h_out, h->d_out, sizeof(float) * (3 * h->T + 2), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(costs_inout, h->d_costs, h->B * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->spilled_traj = h->last.spill_traj != 0;
  h->spilled_cells = h->last.want_cells != 0;
  h->have_rows = true;
  int32_t ff;
  uint32_t fu;
  std::memcpy(&ff, h->h_out + 3 * h->T, 4);
  std::memcpy(&fu, h->h_out + 3 * h->T + 1, 4);
  if (fail_flag_out) {*fail_flag_out = ff;}
  if (furthest_inout) {*furthest_inout = fu;}
  return MPPI_OK;
}

// tuning aid: accumulated host time (ns) of the steady-state call by phase, and the number of calls [7]:
// [0] build_params, [1] stage_costmap, [2] event record, [3] graph launch, [4] event record, [5] wait for the result,
// [6] copy-out + event read-back.  reset != 0 clears the counters.
mppi_status mppi_debug_get_host_ns(mppi_handle * h, uint64_t out8[8], int32_t reset)
{
  if (!h || !out8) {return MPPI_E_CONFIG;}
  for (int i = 0; i < 8; ++i) {out8[i] = h->host_ns[i]; if (reset) {h->host_ns[i] = 0;}}
  return MPPI_OK;
}

// Zero-copy costmap hand-off (SURVEY 8f-4): the caller registers the memory its costmaps live in (Costmap2D::getCharMap()
// of the controller's costmap, once, after configure) as pinned; from then on a costmap inside that range is copied to
// the device straight from the caller's buffer while the call runs - no staging memcpy (160 KB at 400 x 400).
mppi_status mppi_register_costmap_memory(mppi_handle * h, const void * base, uint64_t bytes)
{
  if (!h || !base || bytes == 0) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaHostRegister(const_cast<void *>(base), static_cast<size_t>(bytes), cudaHostRegisterPortable));
  h->pinned_ranges.emplace_back(reinterpret_cast<const char *>(base), static_cast<size_t>(bytes));
  return MPPI_OK;
}

mppi_status mppi_unregister_costmap_memory(mppi_handle * h, const void * base)
{
  if (!h || !base) {return MPPI_E_CONFIG;}
  for (size_t i = 0; i < h->pinned_ranges.size(); ++i) {
    if (h->pinned_ranges[i].first == reinterpret_cast<const char *>(base)) {
      CUDA_TRY(h, cudaSetDevice(h->device));
      CUDA_TRY(h, cudaStreamSynchronize(h->stream));
      CUDA_TRY(h, cudaHostUnregister(const_cast<void *>(base)));
      h->pinned_ranges.erase(h->pinned_ranges.begin() + static_cast<long>(i));
      h->costmap_direct = nullptr;
      return MPPI_OK;
    }
  }
  return fail(h, MPPI_E_STATE, "mppi_unregister_costmap_memory: not a registered base address");
}

mppi_status mppi_set_timing(mppi_handle * h, int32_t enable)
{
  if (!h) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->timing = enable != 0;
  return MPPI_OK;
}

mppi_status mppi_set_profiling(mppi_handle * h, int32_t enable)
{
  if (!h) {return MPPI_E_CONFIG;}
  h->profiling = enable != 0;
  return MPPI_OK;
}

mppi_status mppi_get_profile(mppi_handle * h, float ms_out[4], uint64_t * kernel_launches_total, uint64_t * h2d_bytes, uint64_t * d2h_bytes)
{
  if (!h) {return MPPI_E_CONFIG;}
  if (ms_out) {for (int i = 0; i < 4; ++i) {ms_out[i] = h->prof_ms[i];}}
  if (kernel_launches_total) {*kernel_launches_total = h->launches;}
  if (h2d_bytes) {*h2d_bytes = h->h2d_bytes;}
  if (d2h_bytes) {*d2h_bytes = h->d2h_bytes;}
  return MPPI_OK;
}

// Several shards of ONE optimisation problem driven from one process (one handle per shard, on any mix of
// devices): same two exchanges as the NCCL path, carried by small async copies through pinned host memory.
// This is what a single-process controller (the ROS plugin) uses to spread a large batch over the GPUs of a box,
// and it lets the sharded code path run on a single GPU (two handles on one device) in the tests.
mppi_status mppi_optimize_sharded(mppi_handle ** hs, int32_t n, const mppi_cycle_in * in, mppi_cycle_out * out)
{
  if (!hs || n < 1 || n > kMaxRanks || !in) {return MPPI_E_CONFIG;}
  for (int i = 0; i < n; ++i) {
    if (!hs[i]) {return MPPI_E_CONFIG;}
    if (hs[i]->T != hs[0]->T || hs[i]->cfg.iteration_count != hs[0]->cfg.iteration_count) {
      return fail(hs[i], MPPI_E_CONFIG, "shards must share time_steps and iteration_count");
    }
    if (hs[i]->comm) {return fail(hs[i], MPPI_E_CONFIG, "handle is bound to an NCCL communicator");}
  }
  const int T = hs[0]->T, stride = 3 * T + 2;
  const int words = 1 + kMaxCritics;
  std::vector<unsigned> st_host(static_cast<size_t>(n) * words);
  std::vector<float> partial_host(static_cast<size_t>(n) * stride);
  mppi_status s = MPPI_OK;
  auto on = [&](int i) {cudaSetDevice(hs[i]->device); return hs[i];};
  for (int i = 0; i < n && s == MPPI_OK; ++i) {
    mppi_handle * h = on(i);
    h->nranks = n;   // K3 must not finalize on its own (restored to 1 on every exit path, below)
    if ((s = ensure_gathered(h, n)) != MPPI_OK) {break;}
    if ((s = build_params(h, in, 0, kUnset, true)) != MPPI_OK) {break;}
    if ((s = stage_costmap(h, in->costmap)) != MPPI_OK) {break;}
    if ((s = enqueue_uploads(h)) != MPPI_OK) {break;}
    cudaEventRecord(h->ev0, h->stream);
  }
  for (int it = 0; it < hs[0]->cfg.iteration_count && s == MPPI_OK; ++it) {
    for (int i = 0; i < n && s == MPPI_OK; ++i) {
      mppi_handle * h = on(i);
      s = launch_rollout(h, 0);
      if (s == MPPI_OK && cudaMemcpyAsync(&st_host[static_cast<size_t>(i) * words], h->d_st, words * sizeof(unsigned),
          cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) {s = fail(h, MPPI_E_CUDA, "exchange 1 D2H");}
    }
    // exchange 1: element-wise MAX of (furthest candidate, survivor flags)
    for (int i = 0; i < n && s == MPPI_OK; ++i) {if (cudaStreamSynchronize(on(i)->stream) != cudaSuccess) {s = fail(hs[i], MPPI_E_CUDA, "sync");}}
    for (int w = 0; w < words; ++w) {
      unsigned m = 0;
      for (int i = 0; i < n; ++i) {m = std::max(m, st_host[static_cast<size_t>(i) * words + w]);}
      st_host[w] = m;
    }
    for (int i = 0; i < n && s == MPPI_OK; ++i) {
      mppi_handle * h = on(i);
      if (cudaMemcpyAsync(h->d_st, st_host.data(), words * sizeof(unsigned), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) {
        s = fail(h, MPPI_E_CUDA, "exchange 1 H2D");
        break;
      }
      if ((s = launch_update(h, 0, it)) != MPPI_OK) {break;}
      const int merge_grid = (T + kMergeT - 1) / kMergeT;
      if (h->stream_layout) {
        const int chunks = weighted_sums_chunks(h);
        if ((s = launch_weighted_sums(h)) != MPPI_OK) {break;}
        merge_finalize_kernel<<<merge_grid, kUpdThreads, 0, h->stream>>>(
          reinterpret_cast<const DevParams *>(h->d_params), h->d_partials, chunks, stride, make_bufs(h, 0), 0, h->d_rank_partial, nullptr);
        h->launches++;
      } else if (h->upd_blocks > kLastBlockMergeMax) {
        merge_finalize_kernel<<<merge_grid, kUpdThreads, 0, h->stream>>>(
          reinterpret_cast<const DevParams *>(h->d_params), h->d_partials, h->upd_blocks, stride, make_bufs(h, 0), 0, h->d_rank_partial, nullptr);
        h->launches++;
      }
      if (cudaGetLastError() != cudaSuccess) {s = fail(h, MPPI_E_CUDA, "launch");  break;}
      if (cudaMemcpyAsync(&partial_host[static_cast<size_t>(i) * stride], h->d_rank_partial, stride * sizeof(float),
          cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) {s = fail(h, MPPI_E_CUDA, "exchange 2 D2H");}
    }
    // exchange 2: every shard gets all (min, sum, weighted control sums) records and merges them redundantly
    for (int i = 0; i < n && s == MPPI_OK; ++i) {if (cudaStreamSynchronize(on(i)->stream) != cudaSuccess) {s = fail(hs[i], MPPI_E_CUDA, "sync");}}
    for (int i = 0; i < n && s == MPPI_OK; ++i) {
      mppi_handle * h = on(i);
      if (cudaMemcpyAsync(h->d_gathered, partial_host.data(), static_cast<size_t>(n) * stride * sizeof(float), cudaMemcpyHostToDevice,
          h->stream) != cudaSuccess) {s = fail(h, MPPI_E_CUDA, "exchange 2 H2D"); break;}
      merge_finalize_kernel<<<(T + kMergeT - 1) / kMergeT, kUpdThreads, 0, h->stream>>>(
        reinterpret_cast<const DevParams *>(h->d_params), h->d_gathered, n, stride, make_bufs(h, 0), 1, nullptr, nullptr);
      h->launches++;
      if (cudaGetLastError() != cudaSuccess) {s = fail(h, MPPI_E_CUDA, "launch"); break;}
    }
  }
  if (s != MPPI_OK) {
    // nothing to deliver: drain what was enqueued and hand every shard back as a single-rank handle
    for (int i = 0; i < n; ++i) {
      mppi_handle * h = on(i);
      cudaStreamSynchronize(h->stream);
      h->nranks = 1;
      h->wait_packets = false;
    }
    cudaGetLastError();
    return s;
  }
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = on(i);
    if (s == MPPI_OK) {
      if (cudaMemcpyAsync(h->h_out, h->d_out, sizeof(float) * (3 * T + 2), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) {
        s = fail(h, MPPI_E_CUDA, "result D2H");
      }
      cudaEventRecord(h->ev1, h->stream);
    }
    h->cycle_uploaded = true;
    h->wait_packets = false;   // this path copies its result back (no fused kernel here)
  }
  mppi_status first = s;
  for (int i = 0; i < n; ++i) {
    mppi_handle * h = on(i);
    const mppi_status f = finish_optimize(h, (i == 0 && s == MPPI_OK) ? out : nullptr);
    if (f != MPPI_OK && first == MPPI_OK) {first = f;}
    h->nranks = 1;
  }
  return first;
}

// ---- sharding ------------------------------------------------------------------------------------
mppi_status mppi_comm_get_unique_id(uint8_t id_out[MPPI_NCCL_UNIQUE_ID_BYTES])
{
  std::string err;
  if (!g_nccl.load(err)) {return MPPI_E_NCCL;}
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == MPPI_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId size");
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) {return MPPI_E_NCCL;}
  std::memcpy(id_out, &id, sizeof(id));
  return MPPI_OK;
}

mppi_status mppi_comm_init(mppi_handle * h, const uint8_t id[MPPI_NCCL_UNIQUE_ID_BYTES], int32_t rank, int32_t nranks)
{
  if (!h || !id || nranks < 1 || rank < 0 || rank >= nranks) {return MPPI_E_CONFIG;}
  if (!g_nccl.load(h->err)) {return MPPI_E_NCCL;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof(uid));
  NCCL_TRY(h, g_nccl.CommInitRank(&h->comm, nranks, uid, rank));
  h->rank = rank; h->nranks = nranks;
  return ensure_gathered(h, nranks);
}

// ---- peer-memory exchange: no NCCL, the exchanges ride inside K3 and the merge kernel (mppi_device.cuh PeerComm) ----
mppi_status mppi_comm_get_mailbox_handle(mppi_handle * h, uint8_t handle_out[MPPI_IPC_HANDLE_BYTES])
{
  static_assert(sizeof(cudaIpcMemHandle_t) == MPPI_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  if (!h || !handle_out) {return MPPI_E_CONFIG;}
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (!h->d_mailbox) {
    CUDA_TRY(h, cudaMalloc(&h->d_mailbox, sizeof(unsigned) * kBoxWords));
    CUDA_TRY(h, cudaMemset(h->d_mailbox, 0, sizeof(unsigned) * kBoxWords));
  }
  cudaIpcMemHandle_t ipc;
  CUDA_TRY(h, cudaIpcGetMemHandle(&ipc, h->d_mailbox));
  std::memcpy(handle_out, &ipc, sizeof(ipc));
  return MPPI_OK;
}

mppi_status mppi_comm_connect_peers(mppi_handle * h, const uint8_t * handles, int32_t rank, int32_t nranks)
{
  if (!h || !handles || nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks) {return MPPI_E_CONFIG;}
  if (!h->d_mailbox) {return fail(h, MPPI_E_STATE, "mppi_comm_get_mailbox_handle first");}
  if (h->comm) {return fail(h, MPPI_E_STATE, "handle is bound to an NCCL communicator");}
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  drop_graphs(h);
  for (int r = 0; r < nranks; ++r) {
    if (r == rank) {h->peer_box[r] = h->d_mailbox; continue;}
    cudaIpcMemHandle_t ipc;
    std::memcpy(&ipc, handles + static_cast<size_t>(r) * MPPI_IPC_HANDLE_BYTES, sizeof(ipc));
    void * p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(h, MPPI_E_CUDA, std::string("cudaIpcOpenMemHandle (peer access between the GPUs of the box is required): ") + cudaGetErrorString(e));
    }
    h->peer_box[r] = static_cast<uint2 *>(p);
  }
  h->rank = rank; h->nranks = nranks; h->peer_mode = nranks > 1;
  return MPPI_OK;
}

mppi_status mppi_comm_destroy(mppi_handle * h)
{
  if (!h) {return MPPI_E_CONFIG;}
  if (h->peer_mode) {
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    drop_graphs(h);
    for (int r = 0; r < h->nranks; ++r) {
      if (r != h->rank && h->peer_box[r]) {cudaIpcCloseMemHandle(h->peer_box[r]);}
      h->peer_box[r] = nullptr;
    }
    h->peer_mode = false;
  }
  if (h->comm) {
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    g_nccl.CommDestroy(h->comm);
    h->comm = nullptr;
  }
  h->rank = 0; h->nranks = 1;
  return MPPI_OK;
}

}  // extern "C"
