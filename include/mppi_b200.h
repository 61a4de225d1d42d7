/*
 * mppi_b200.h -- C ABI of the B200-native MPPI optimisation loop.
 *
 * This is the drop-in boundary for the hot path of nav2_sortham_controller (the MPPI controller of
 * soham2560/MPCHoloNavigation).  A shared library exporting these symbols replaces the body of
 * sortham::Optimizer (reference: include/nav2_sortham_controller/optimizer.hpp:72-117) and of the
 * built-in critic plugins; the nav2_core::Controller plugin, the pluginlib critic classes and the ROS
 * parameter surface stay on the host (see INTEGRATION.md for the shim).
 *
 * Conventions
 *  - plain C, POD structs, pointers and sizes only; no exceptions cross the boundary: every call returns
 *    an mppi_status and mppi_last_error() gives the text of the last failure on that handle;
 *  - all [B,T] planes are float32, row-major (b major, t minor), exactly the xtensor layout of the
 *    reference (models/state.hpp:30-56); [T] and [N] vectors are float32;
 *  - the caller owns every input buffer for the duration of the call only; the library copies what it
 *    needs (pinned staging + async copies) before returning (a device-resident costmap is read in place, see
 *    mppi_set_costmap_residency);
 *  - a handle is externally synchronised and non-re-entrant (the reference holds the parameter and
 *    costmap mutexes around evalControl, src/controller.cpp:94-103); distinct handles are independent;
 *  - there is NO CPU fallback: if no CUDA device is usable the calls fail with MPPI_E_CUDA.
 *
 * "ref:" comments cite the reference interface each entry point replaces, relative to
 * /root/reference/nav2_sortham_controller/.
 */
#ifndef MPPI_B200_H_
#define MPPI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPPI_ABI_VERSION 1

typedef enum mppi_status {
  MPPI_OK = 0,
  MPPI_E_CONFIG = 1,   /* invalid argument / configuration (ref: std::runtime_error in setMotionModel, optimizer.cpp:421-424) */
  MPPI_E_CUDA = 2,     /* CUDA runtime failure, or no device */
  MPPI_E_NCCL = 3,     /* communicator failure (sharded configurations only) */
  MPPI_E_STATE = 4     /* call made in the wrong order (e.g. getter before any optimize) */
} mppi_status;

typedef enum mppi_motion_model {   /* ref: optimizer.cpp:412-426, motion_models.hpp:85-171 */
  MPPI_MODEL_DIFF_DRIVE = 0,
  MPPI_MODEL_OMNI = 1,
  MPPI_MODEL_ACKERMANN = 2
} mppi_motion_model;

/* Critic kinds: one per class of critics.xml:1-53 (same order as the plugin names sort). */
typedef enum mppi_critic_kind {
  MPPI_CRITIC_CONSTRAINT = 0,        /* sortham::critics::ConstraintCritic       src/critics/constraint_critic.cpp */
  MPPI_CRITIC_COST = 1,              /* sortham::critics::CostCritic             src/critics/cost_critic.cpp */
  MPPI_CRITIC_GOAL = 2,              /* sortham::critics::GoalCritic             src/critics/goal_critic.cpp */
  MPPI_CRITIC_GOAL_ANGLE = 3,        /* sortham::critics::GoalAngleCritic        src/critics/goal_angle_critic.cpp */
  MPPI_CRITIC_OBSTACLES = 4,         /* sortham::critics::ObstaclesCritic        src/critics/obstacles_critic.cpp */
  MPPI_CRITIC_PATH_ALIGN = 5,        /* sortham::critics::PathAlignCritic        src/critics/path_align_critic.cpp */
  MPPI_CRITIC_PATH_ALIGN_LEGACY = 6, /* sortham::critics::PathAlignLegacyCritic  src/critics/path_align_legacy_critic.cpp */
  MPPI_CRITIC_PATH_ANGLE = 7,        /* sortham::critics::PathAngleCritic        src/critics/path_angle_critic.cpp */
  MPPI_CRITIC_PATH_FOLLOW = 8,       /* sortham::critics::PathFollowCritic       src/critics/path_follow_critic.cpp */
  MPPI_CRITIC_PREFER_FORWARD = 9,    /* sortham::critics::PreferForwardCritic    src/critics/prefer_forward_critic.cpp */
  MPPI_CRITIC_TWIRLING = 10,         /* sortham::critics::TwirlingCritic         src/critics/twirling_critic.cpp */
  MPPI_CRITIC_VELOCITY_DEADBAND = 11,/* sortham::critics::VelocityDeadbandCritic src/critics/velocity_deadband_critic.cpp */
  MPPI_CRITIC_KIND_COUNT = 12
} mppi_critic_kind;

#define MPPI_MAX_CRITICS 16
#define MPPI_MAX_FOOTPRINT 32
#define MPPI_MAX_TIME_STEPS 256
#define MPPI_MAX_PATH_POINTS 1024

/* Optimizer settings. ref: Optimizer::getParams optimizer.cpp:62-93, models/optimizer_settings.hpp:28-41.
 * Field names are the ROS parameter names; defaults (mppi_config_default) are the reference's. */
typedef struct mppi_config {
  int32_t batch_size;        /* "batch_size" 1000  (the LOCAL share when sharded, see shard_*) */
  int32_t time_steps;        /* "time_steps" 56 */
  int32_t iteration_count;   /* "iteration_count" 1 */
  float model_dt;            /* "model_dt" 0.05 */
  float temperature;         /* "temperature" 0.3 */
  float gamma;               /* "gamma" 0.015 */
  float vx_max, vx_min, vy_max, wz_max;   /* base constraints 0.5 / -0.35 / 0.5 / 1.9 */
  float vx_std, vy_std, wz_std;           /* sampling std 0.2 / 0.2 / 0.4 */
  int32_t motion_model;      /* mppi_motion_model; reference default "DiffDrive" */
  float ackermann_min_turning_r;  /* "AckermannConstraints.min_turning_r" 0.2 (motion_models.hpp:93-94) */
  int32_t regenerate_noises; /* "regenerate_noises" false (noise_generator.cpp:35) */
  uint64_t seed;             /* Philox key; the reference's engine is unseeded (noise_generator.cpp:107-122) */
  int32_t device;            /* CUDA device ordinal */
  /* sharding of one optimisation problem over several handles/GPUs (SURVEY 8e): this handle owns the
   * global trajectories [shard_offset, shard_offset + batch_size) of shard_total.  Single GPU: 0 / 0. */
  int64_t shard_offset;
  int64_t shard_total;
} mppi_config;

/* One critic of the "critics" list, in list order (critic_manager.cpp:39-60).  Flat on purpose: every
 * parameter any built-in critic reads has a field; a critic ignores the fields it does not own.
 * Defaults per kind: mppi_critic_default(). */
typedef struct mppi_critic_desc {
  int32_t kind;                    /* mppi_critic_kind */
  int32_t enabled;                 /* "<critic>.enabled" true (critic_function.hpp:81) */
  uint32_t cost_power;             /* "cost_power" 1 */
  float cost_weight;               /* "cost_weight"; CostCritic: raw value, divided by 254 inside (cost_critic.cpp:34) */
  float threshold_to_consider;     /* Goal 1.4, GoalAngle 0.5, PreferForward 0.5, PathAlign* 0.5, PathFollow 1.4, PathAngle 0.5 */
  int32_t offset_from_furthest;    /* PathAlign* 20, PathFollow 6, PathAngle 4 */
  int32_t trajectory_point_step;   /* PathAlign* 4 */
  float max_path_occupancy_ratio;  /* PathAlign* 0.07 */
  int32_t use_path_orientations;   /* PathAlign* false */
  float max_angle_to_furthest;     /* PathAngle 1.2 */
  int32_t forward_preference;      /* PathAngle true */
  int32_t consider_footprint;      /* Cost false, Obstacles false */
  float collision_cost;            /* Cost 1e6, Obstacles 1e4 */
  float critical_cost;             /* Cost 300 */
  float near_goal_distance;        /* Cost 0.5, Obstacles 0.5 */
  float repulsion_weight;          /* Obstacles 1.5 */
  float critical_weight;           /* Obstacles 20 */
  float collision_margin_distance; /* Obstacles 0.10 */
  float cost_scaling_factor;       /* Obstacles 10.0 (read only if an inflation layer exists, obstacles_critic.cpp:78-80) */
  float inflation_radius;          /* Obstacles 0.55 (same) */
  float deadband_velocities[3];    /* VelocityDeadband {0,0,0} */
} mppi_critic_desc;

/* What the critics need to know about the layered costmap and the robot footprint.
 * ref: Costmap2DROS::getRobotFootprint, LayeredCostmap::getInscribedRadius/getCircumscribedRadius/
 * isTrackingUnknown, InflationLayer::computeCost (call sites obstacles_critic.cpp:53-97,102,188,219;
 * cost_critic.cpp:63-106,178,185). */
typedef struct mppi_robot_desc {
  int32_t footprint_size;                    /* number of polygon vertices (<= MPPI_MAX_FOOTPRINT) */
  double footprint_x[MPPI_MAX_FOOTPRINT];    /* vertices in the robot frame */
  double footprint_y[MPPI_MAX_FOOTPRINT];
  double inscribed_radius;
  double circumscribed_radius;
  int32_t inflation_layer_found;             /* an InflationLayer is among the costmap plugins */
  double inflation_cost_scaling_factor;      /* the LAYER's cost_scaling_factor (used by computeCost) */
  int32_t track_unknown;                     /* LayeredCostmap::isTrackingUnknown() */
} mppi_robot_desc;

/* Costmap2D view for one cycle. ref: nav2_costmap_2d::Costmap2D (getCharMap, getSizeInCellsX/Y,
 * getResolution, getOriginX/Y), read under the costmap mutex at controller.cpp:99-100. */
typedef struct mppi_costmap {
  const uint8_t * cells;     /* size_y rows of size_x bytes; index = my * size_x + mx.  Host memory, or device memory
                                of the handle's device after mppi_set_costmap_residency(h, MPPI_COSTMAP_DEVICE) */
  uint32_t size_x, size_y;
  double resolution;
  double origin_x, origin_y;
} mppi_costmap;

/* Per-cycle inputs of Optimizer::evalControl -> prepare (optimizer.cpp:134-141,185-204). */
typedef struct mppi_cycle_in {
  double pose_x, pose_y;     /* robot_pose.pose.position */
  double pose_yaw;           /* tf2::getYaw(robot_pose.pose.orientation) */
  double speed_vx, speed_vy, speed_wz;   /* robot_speed.linear.x/.y, angular.z */
  double goal_x, goal_y;     /* goal.position */
  double goal_checker_xy_tolerance;      /* GoalChecker::getTolerances pose_tolerance.position.x; < 0 when goal_checker == nullptr */
  int32_t path_size;         /* N (<= MPPI_MAX_PATH_POINTS) */
  const float * path_x;      /* utils::toTensor(plan) (utils.hpp:180-192) */
  const float * path_y;
  const float * path_yaw;
  mppi_costmap costmap;
} mppi_cycle_in;

/* Outputs of one optimize() (optimizer.cpp:157-164): the clipped mean control sequence and the
 * "all trajectories collide" flag that drives Optimizer::fallback (optimizer.cpp:166-183). */
typedef struct mppi_cycle_out {
  float * control_vx;        /* [T], caller-provided, may be NULL */
  float * control_vy;
  float * control_wz;
  int32_t fail_flag;         /* CriticData::fail_flag after the last iteration */
  uint32_t furthest_reached_path_point;  /* CriticData::furthest_reached_path_point, UINT32_MAX if unset */
  float device_ms;           /* CUDA-event time of the kernels of this call (and of the copies that are part of the
                                captured cycle); 0 when mppi_set_timing(h, 0) */
} mppi_cycle_out;

/* Cycle inputs of a bound group (mppi_optimize_group_device), in device memory of the group's device, one row per member
 * in bind order: what mppi_cycle_in carries besides the costmap. */
typedef struct mppi_group_inputs {
  const double * state;      /* [n][8]: pose_x, pose_y, pose_yaw, speed_vx, speed_vy, speed_wz, goal_x, goal_y */
  const double * goal_checker_xy_tolerance;   /* [n]; < 0: goal_checker == nullptr */
  const int32_t * path_size; /* [n]; each in [1, MPPI_MAX_PATH_POINTS] and <= path_stride */
  const float * path;        /* [n][3][path_stride]: x, y, yaw */
  int32_t path_stride;       /* >= every path_size */
} mppi_group_inputs;

typedef struct mppi_handle mppi_handle;

/* ---- life cycle (ref: Optimizer::initialize/shutdown/reset optimizer.cpp:35-60,116-132) ---- */
void mppi_config_default(mppi_config * cfg);
void mppi_critic_default(int32_t kind, mppi_critic_desc * desc);
mppi_status mppi_create(const mppi_config * cfg, mppi_handle ** out);
void mppi_destroy(mppi_handle * h);
/* reset(): zero control sequence and costs, restore base constraints, redraw the noise */
mppi_status mppi_reset(mppi_handle * h);
const char * mppi_last_error(const mppi_handle * h);
int32_t mppi_abi_version(void);

/* ---- configuration ---- */
/* ref: CriticManager::loadCritics critic_manager.cpp:42-60 + each critic's initialize() */
mppi_status mppi_set_critics(mppi_handle * h, const mppi_critic_desc * critics, int32_t n);
mppi_status mppi_set_robot(mppi_handle * h, const mppi_robot_desc * robot);
/* ref: Optimizer::setSpeedLimit optimizer.cpp:428-453 (speed_limit == 0 means NO_SPEED_LIMIT) */
mppi_status mppi_set_speed_limit(mppi_handle * h, double speed_limit, int32_t percentage);
/* current (speed-limited) constraints: vx_max, vx_min, vy, wz */
mppi_status mppi_get_constraints(const mppi_handle * h, float out4[4]);

/* ---- noise (ref: NoiseGenerator noise_generator.cpp:65-122) ---- */
/* parity mode: inject the reference's noise tensors, [B,T] row-major each; vy may be NULL (zeros) */
mppi_status mppi_set_noise(mppi_handle * h, const float * vx, const float * vy, const float * wz);
/* Philox4x32-10 + Box-Muller kernel; counter = (global b, t/4, plane, stream) so shards tile exactly */
mppi_status mppi_generate_noise(mppi_handle * h, uint64_t stream);
mppi_status mppi_get_noise(mppi_handle * h, float * vx, float * vy, float * wz);

/* ---- warm-start state (ref: control_sequence_ optimizer.hpp:250) ---- */
mppi_status mppi_set_control_sequence(mppi_handle * h, const float * vx, const float * vy, const float * wz);
mppi_status mppi_get_control_sequence(mppi_handle * h, float * vx, float * vy, float * wz);
/* ref: Optimizer::shiftControlSequence optimizer.cpp:206-225 */
mppi_status mppi_shift_control_sequence(mppi_handle * h);

/* ---- where the cycle's costmap lives ---- */
/* MPPI_COSTMAP_HOST (default): costmap.cells of every cycle entry point is host memory; the library stages and copies it.
 * MPPI_COSTMAP_DEVICE: costmap.cells is device memory of the handle's device (a GPU costmap producer, a map shared by a
 * fleet); the map is read in place, never copied, and the path-validity tables that depend on it are made on the device.
 * Applies to mppi_optimize, mppi_eval_control, mppi_upload_cycle (+ mppi_optimize_resident), mppi_optimize_batch[_resident]
 * (bound or not; members choose independently and may share one map) and mppi_optimize_sharded (every handle must be on
 * the map's device).  The geometry fields keep their meaning.  Contract:
 *  - the map's contents are complete before the call (the library does not wait on the caller's streams);
 *  - the map stays unchanged until the call that consumes it returns: for mppi_upload_cycle, the mppi_optimize_resident
 *    that follows;
 *  - nothing reads the map after that call returns (the regenerate_noises redraw behind the result does not);
 *  - the pointer may differ in every cycle.
 * The pointer is checked before anything is enqueued: host, managed or another device's memory, or an allocation smaller
 * than size_x * size_y, fails with MPPI_E_CONFIG.  The last pointer that passed is remembered and not checked again while
 * the map's size does not grow: an address that is freed and handed out again must not come back with an allocation
 * smaller than the map (mppi_set_costmap_residency forgets the remembered pointer).  A failed mppi_upload_cycle in device
 * mode leaves nothing to run: mppi_optimize_resident then fails with MPPI_E_STATE.  mppi_optimize_sharded needs every
 * shard in the same residency.  mppi_integrate_state_velocities keeps working (it needs no map);
 * mppi_score_trajectories takes host maps only and fails with MPPI_E_CONFIG in device mode. */
#define MPPI_COSTMAP_HOST 0
#define MPPI_COSTMAP_DEVICE 1
mppi_status mppi_set_costmap_residency(mppi_handle * h, int32_t residency);

/* ---- the hot path ---- */
/* prepare() + optimize() (optimizer.cpp:141-145 without the fallback loop, which stays in the host
 * mirror because it throws): costs are zeroed, then iteration_count x {noised rollout, critics,
 * softmax update}.  Host buffers in (the costmap may be device memory: mppi_set_costmap_residency), host buffers out. */
mppi_status mppi_optimize(mppi_handle * h, const mppi_cycle_in * in, mppi_cycle_out * out);
/* Optimizer::evalControl (optimizer.cpp:134-155) for one attempt: prepare() + optimize() and, if fail_flag stayed clear,
 * utils::savitskyGolayFilter (utils.hpp:442-605), getControlFromSequenceAsTwist (optimizer.cpp:396-410) and, when
 * shift_control_sequence != 0 (Optimizer::setOffset, optimizer.cpp:95-114), shiftControlSequence (:206-225) -- all on
 * the device, so the warm-start sequence and the 4-deep control history never leave it.  cmd_out = (vx, vy, wz) of
 * the returned twist (vy = 0 for non-holonomic models).  When out->fail_flag is set nothing after optimize() ran:
 * the caller does what Optimizer::fallback does (mppi_reset, retry up to retry_attempt_limit, then throw). */
mppi_status mppi_eval_control(mppi_handle * h, const mppi_cycle_in * in, int32_t shift_control_sequence,
                              mppi_cycle_out * out, float cmd_out[3]);
/* control_history_ (optimizer.hpp:251): [4][3] = (vx, vy, wz) of the last four commands, oldest first */
mppi_status mppi_set_control_history(mppi_handle * h, const float hist12[12]);
mppi_status mppi_get_control_history(mppi_handle * h, float hist12[12]);
/* batched multi-robot form: n independent handles (possibly on several devices) launched back to back
 * and then joined, so their kernels overlap */
mppi_status mppi_optimize_batch(mppi_handle ** hs, const mppi_cycle_in * ins, mppi_cycle_out * outs, int32_t n);
/* Multi-robot server (BASELINE configs[4]): bind n unsharded handles of ONE device into a group.  Members may differ in
 * batch_size and time_steps (robot types with their own horizon; a handle re-created after a parameter change binds
 * back with the others).  A host-resident costmap travels in the member's slice of the group's upload buffer (at least
 * 64 KB, or the largest member's staging capacity at bind time); a device-resident one (mppi_set_costmap_residency) stays
 * where it is, whatever its size, and several members may point at the same map.  The members move to the stream layout and share the first handle's stream from then on, and
 * mppi_optimize_batch[_resident] over exactly this group, in this order, runs in chunks of up to 64 robots: each chunk is
 * one strided upload plus four kernel launches per iteration, each launch sized for the chunk's largest member.  Members
 * with regenerate_noises redraw their noise in
 * batched launches too (between iterations per chunk, and once for the whole group behind the last chunk's results), and
 * continue the same Philox stream sequence after mppi_batch_unbind.  Every other call keeps working on a bound handle; a
 * cycle whose members do not all qualify (evalControl tail, profiling, members with different iteration_count, ...) runs
 * them one by one.  Destroying a member dissolves the group. */
mppi_status mppi_batch_bind(mppi_handle ** handles, int32_t n);
mppi_status mppi_batch_unbind(mppi_handle * any_member);
/* The same over inputs already resident on the device (mppi_upload_cycle on every handle).  Measurement hook. */
mppi_status mppi_optimize_batch_resident(mppi_handle ** handles, mppi_cycle_out * outs, int32_t n);
/* Device time of the last batch call over these handles (one device, timing on): first start event to latest end
 * event; the handles run concurrently on their own streams, so their device_ms overlap. */
mppi_status mppi_batch_span_ms(mppi_handle ** handles, int32_t n, float * ms_out);
/* mppi_optimize_batch over exactly a bound group (bind order) whose cycle inputs are already in device memory: a GPU
 * simulator's state tensors, or a fleet server's one packed upload.  Every member must be in MPPI_COSTMAP_DEVICE mode and
 * qualify for the group's batched launches.  maps[n] are HOST descriptors whose cells point into device memory (checked
 * as for mppi_set_costmap_residency); outs as for mppi_optimize_batch.  The members' cycle records are built on the
 * device, so the host does no per-robot work besides the job table; the result is bit for bit what mppi_optimize_batch
 * returns for the same inputs (one exception, DESIGN.md section 2: PathAngle's gate for a path point within 1e-5 of the
 * threshold's cosine is decided with the device's atan2f).
 * Contract, as for a device costmap: the inputs are complete before the call, stay unchanged until it returns, and
 * nothing reads them afterwards (the caller synchronises its own streams first).
 * MPPI_E_CONFIG before anything is enqueued: hs is not exactly a bound group, a member is in host-costmap mode or does not
 * qualify (evalControl tail, profiling, another iteration_count than member 0; there is no one-by-one fallback), both
 * PathAlign critics enabled with different trajectory_point_step, an input pointer is not device memory of the group's
 * device or its allocation holds fewer than n rows, a map is rejected.
 * A path_size outside [1, min(MPPI_MAX_PATH_POINTS, path_stride)] is seen on the device: that member's launches are
 * cancelled, its outputs and warm start (control sequence, costs, noise) stay as they were, the other members run, and the
 * call returns MPPI_E_CONFIG with the member's index in mppi_last_error(hs[0]).  The call leaves a staged cycle for
 * mppi_optimize_batch_resident like mppi_optimize_batch does (not for a member that failed). */
mppi_status mppi_optimize_group_device(mppi_handle ** hs, int32_t n, const mppi_group_inputs * in,
                                       const mppi_costmap * maps, mppi_cycle_out * outs);
/* Test hook: the first `capacity` bytes of the device copy of the handle's last cycle record (record + path tail), its
 * meaningful length in *record_bytes, and in *angle_band_hits the number of PathAngle gate decisions the device inputs
 * of mppi_optimize_group_device have left to the device's atan2f since create (a path point exactly under the robot is
 * not counted: atan2f(0, 0) = 0 on either side). */
mppi_status mppi_debug_get_record(mppi_handle * h, void * out, uint64_t capacity, uint64_t * record_bytes,
                                  uint64_t * angle_band_hits);

/* Split-phase form for data already resident on the device (bench "value" leg, CUDA-graph replay):
 * upload once, then run the device part only.  A device-resident costmap is read by mppi_optimize_resident: it must stay
 * unchanged until that call returns. */
mppi_status mppi_upload_cycle(mppi_handle * h, const mppi_cycle_in * in);
mppi_status mppi_optimize_resident(mppi_handle * h, mppi_cycle_out * out);

/* ---- introspection of the last optimize (debug / parity / visualisation) ---- */
/* request materialisation: bit 0 trajectories x,y,yaw [B,T]; bit 1 costmap cell index per (b,t)
 * (int32 my*size_x+mx, -1 off-map); bit 2 per-critic cost rows.  Off by default (extra HBM traffic). */
#define MPPI_WANT_TRAJECTORIES 1u
#define MPPI_WANT_CELLS 2u
#define MPPI_WANT_CRITIC_COSTS 4u
mppi_status mppi_set_outputs(mppi_handle * h, uint32_t want_mask);
/* ref: Optimizer::getGeneratedTrajectories optimizer.cpp:455-458 */
mppi_status mppi_get_trajectories(mppi_handle * h, float * x, float * y, float * yaw);
/* ref: the only consumer of the candidate trajectories, TrajectoryVisualizer::add (trajectory_visualizer.cpp:86-108), draws
 * x(i, j), y(i, j) for i = 0, trajectory_step, ... and j = 0, time_step, ... ("TrajectoryVisualizer.trajectory_step" 5,
 * ".time_step" 3): K2 materialises exactly that lattice.  (0, 0) switches it off.  Outputs are
 * [ceil(B / trajectory_step)][ceil(T / time_step)] row-major. */
mppi_status mppi_set_visualization(mppi_handle * h, int32_t trajectory_step, int32_t time_step);
mppi_status mppi_get_visualization(mppi_handle * h, float * x, float * y);
mppi_status mppi_get_cells(mppi_handle * h, int32_t * cells);
/* total costs_[B] after the last iteration (before they are consumed by the softmax: includes gamma term) */
mppi_status mppi_get_costs(mppi_handle * h, float * costs);
/* contribution of critic `index` (list order) in the last iteration, [B] */
mppi_status mppi_get_critic_costs(mppi_handle * h, int32_t index, float * costs);
/* ref: Optimizer::getOptimizedTrajectory optimizer.cpp:345-360 -> [T,3] (x, y, yaw) */
mppi_status mppi_get_optimized_trajectory(mppi_handle * h, double pose_x, double pose_y, double pose_yaw, float * traj_t3);

/* ---- critic-level and rollout-level entry points (what the reference's unit tests call) ---- */
/* ref: Optimizer::integrateStateVelocities(Trajectories&, const State&) optimizer.cpp:313-343:
 * state velocities vx,vy,wz [B,T] -> x,y,yaw [B,T] */
mppi_status mppi_integrate_state_velocities(mppi_handle * h, double pose_x, double pose_y, double pose_yaw,
                                            const float * vx, const float * vy, const float * wz,
                                            float * x, float * y, float * yaw);
/* ref: CriticManager::evalTrajectoriesScores(CriticData&) critic_manager.cpp:67-76 on caller-provided
 * State (vx,vy,wz) and Trajectories (x,y,yaw), all [B,T]; costs_inout [B] is accumulated into.
 * furthest_inout: pass UINT32_MAX for "unset" (std::nullopt); returns the value after scoring. */
mppi_status mppi_score_trajectories(mppi_handle * h, const mppi_cycle_in * in,
                                    const float * vx, const float * vy, const float * wz,
                                    const float * x, const float * y, const float * yaw,
                                    float * costs_inout, uint32_t * furthest_inout, int32_t * fail_flag_out);

/* Zero-copy costmap hand-off (ref: the reference reads Costmap2D::getCharMap() in place under the costmap mutex,
 * controller.cpp:99-100).  Register the memory the caller's costmaps live in (cudaHostRegister) once; from then on a
 * costmap inside such a range is copied to the device straight from the caller's buffer during the call, without the
 * staging memcpy.  Costmaps small enough for the fused kernel's own upload (<= 96 KB) keep going through staging. */
mppi_status mppi_register_costmap_memory(mppi_handle * h, const void * base, uint64_t bytes);
mppi_status mppi_unregister_costmap_memory(mppi_handle * h, const void * base);

/* ---- measurement hooks (bench.py: roofline of the dominant kernel, launch count) ---- */
/* when enabled, CUDA events bracket each kernel of optimize() on the handle's stream (adds ~1 us per event) */
mppi_status mppi_set_profiling(mppi_handle * h, int32_t enable);
/* device_ms of mppi_cycle_out costs two event records and an event read-back per call (~5 us of host time); the
 * controller does not need it (the reference has no such output): enable = 0 switches it off, device_ms then reads 0.
 * Default: on. */
mppi_status mppi_set_timing(mppi_handle * h, int32_t enable);
/* last optimize(), summed over iteration_count: ms_out[0] K2 rollout_score, [1] K3 path_softmax_update,
 * [2] exchanges + K4 merge (sharded only), [3] whole device span.  When the fused small-batch kernel ran (one launch
 * for rollout, critics, update and merge) all of it is reported in [0] and [1] = [2] = 0.  kernel_launches_total counts every
 * kernel this handle has launched since create; h2d/d2h are the bytes copied by the last mppi_optimize(). */
mppi_status mppi_get_profile(mppi_handle * h, float ms_out[4], uint64_t * kernel_launches_total,
                             uint64_t * h2d_bytes, uint64_t * d2h_bytes);

/* ---- sharding over GPUs (SURVEY 8e) ---- */
/* single process: n handles (one per shard, cfg.shard_offset / shard_total set, any mix of devices; with a device-resident
 * costmap every handle on the map's device) solve ONE problem; the two tiny exchanges (furthest path point + survivor flags; softmax partials) go through pinned
 * host memory.  Every handle ends with the same control sequence; `out` is filled from hs[0]. */
mppi_status mppi_optimize_sharded(mppi_handle ** hs, int32_t n, const mppi_cycle_in * in, mppi_cycle_out * out);
/* one process per GPU: one handle per rank, the same exchanges as one ncclAllReduce(MAX) and one ncclAllGather */
#define MPPI_NCCL_UNIQUE_ID_BYTES 128
mppi_status mppi_comm_get_unique_id(uint8_t id_out[MPPI_NCCL_UNIQUE_ID_BYTES]);
mppi_status mppi_comm_init(mppi_handle * h, const uint8_t id[MPPI_NCCL_UNIQUE_ID_BYTES], int32_t rank, int32_t nranks);
/* one process per GPU, NO NCCL: the two exchanges go through small mailboxes in peer-mapped HBM (CUDA IPC over NVLink /
 * NVSwitch) and are fused into the kernels on either side of them (remote stores + system-scope flags; consumers spin
 * on local memory, bounded).  Every rank: mppi_comm_get_mailbox_handle -> all-gather the 64-byte handles by any means
 * (MPI, torch.distributed, a file) -> mppi_comm_connect_peers(all handles in rank order).  Needs peer access between
 * the GPUs; MPPI_E_NCCL from mppi_optimize means a rank never arrived (time-out), not a hang. */
#define MPPI_IPC_HANDLE_BYTES 64
mppi_status mppi_comm_get_mailbox_handle(mppi_handle * h, uint8_t handle_out[MPPI_IPC_HANDLE_BYTES]);
mppi_status mppi_comm_connect_peers(mppi_handle * h, const uint8_t * handles /* [nranks][64] */, int32_t rank, int32_t nranks);
mppi_status mppi_comm_destroy(mppi_handle * h);

#ifdef __cplusplus
}
#endif
#endif  /* MPPI_B200_H_ */
