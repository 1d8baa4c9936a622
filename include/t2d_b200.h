/*
 * t2d_b200.h - C ABI of the B200-native batched env.step() hot path for tactics2d.
 *
 * The reference (WoodOxen/tactics2d, pure Python) has no FFI layer: its boundary for
 * this path is five duck-typed Python interfaces.  This library is what a ctypes
 * binding behind those interfaces calls; every entry point names the reference
 * interface it replaces (paths relative to the reference root):
 *
 *   t2d_physics_step     PhysicsModelBase.step            tactics2d/physics/physics_model_base.py:27-38
 *                        SingleTrackKinematics.step       tactics2d/physics/single_track_kinematics.py:178-198
 *                        SingleTrackDynamics.step         tactics2d/physics/single_track_dynamics.py:231-251
 *                        PointMass.step                   tactics2d/physics/point_mass.py:209-232
 *   t2d_set_type_table   ParticipantBase / templates      tactics2d/participant/element/participant_template.py:42-257,
 *                                                         vehicle.py:111-118,179-221, cyclist.py:76-94, pedestrian.py:70-88
 *   t2d_set_map          StaticCollision.reset / OutBound.reset
 *                                                         tactics2d/traffic/event_detection/collision.py:45-46, out_bound.py:50-65
 *   t2d_bind_wheel_state the omega_wf / omega_wr arguments of SingleTrackDrift.step
 *                                                         tactics2d/physics/single_track_drift.py:467-499
 *   t2d_bind_state       Trajectory.add_state / current state
 *                                                         tactics2d/participant/trajectory/trajectory.py:115-149
 *   t2d_step             ScenarioManager.update + check_status
 *                                                         tactics2d/traffic/scenario_manager.py:63-73,
 *                                                         tactics2d/envs/parking.py:352-392 (tick), :243-248 (done rule)
 *                        ParticipantBase.get_pose         tactics2d/participant/element/vehicle.py:263-281
 *                        DynamicCollision.update          tactics2d/traffic/event_detection/collision.py:18-25
 *                        StaticCollision.update           tactics2d/traffic/event_detection/collision.py:37-43
 *                        OutBound.update                  tactics2d/traffic/event_detection/out_bound.py:37-48
 *                        TimeExceed.update                tactics2d/traffic/event_detection/time_exceed.py:26-33
 *   t2d_set_goal         Arrival.update / NoAction.update  tactics2d/traffic/event_detection/arrival.py:32-47, no_action.py:32-53
 *   t2d_lidar_scan       SingleLineLidar._scan_obstacles   tactics2d/sensor/lidar.py:128-221
 *   t2d_set_controllers  IDMController / AccelerationController / PurePursuitController objects
 *                                                         tactics2d/controller/idm_controller.py:33-58,
 *                                                         acceleration_controller.py:33-80, pure_pursuit_controller.py:26-49
 *   t2d_set_paths        the `waypoints` LineString of PurePursuitController.step   pure_pursuit_controller.py:76,92
 *   t2d_control          ControllerBase.step for every controlled participant
 *                                                         idm_controller.py:59-141, acceleration_controller.py:82-145,
 *                                                         pure_pursuit_controller.py:51-98
 *   t2d_check_events     the same detectors on caller-supplied poses (no physics)
 *   t2d_reset            ScenarioManager.reset / ParticipantBase.reset
 *                                                         tactics2d/envs/parking.py:397-441, participant_base.py:236-246
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the ABI;
 *   - every function returns 0 on success or a negative T2D_E_* code; the message of the
 *     last error on the calling thread is t2d_last_error(); no exception crosses;
 *   - all array arguments of t2d_step / t2d_check_events / t2d_reset / t2d_physics_step are
 *     DEVICE pointers owned by the caller (PyTorch tensors' data_ptr()); the library never
 *     allocates or frees them.  t2d_set_type_table / t2d_set_map take HOST pointers and copy;
 *   - work is enqueued on the cudaStream_t passed as `stream` (NULL = legacy default
 *     stream) and the call returns without a host synchronisation;
 *   - a context belongs to one device and is not thread-safe.
 *
 * Layout: structure-of-arrays, scenario-major.  Participant (n, m) of an N x M world lives
 * at index n*M + m of every [N, M] array.  fp32 state, uint8 type ids, int16 hit indices.
 */
#ifndef T2D_B200_H
#define T2D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define T2D_VERSION 100 /* 0.1.0 */

/* error codes */
#define T2D_OK 0
#define T2D_E_INVALID (-1)     /* bad argument */
#define T2D_E_CUDA (-2)        /* a CUDA runtime call failed; see t2d_last_error() */
#define T2D_E_UNSUPPORTED (-3) /* configuration outside what the kernels cover */
#define T2D_E_STATE (-4)       /* call order: state not bound, type table not set ... */

/* physics model ids (t2d_type_params.model) */
#define T2D_MODEL_KINEMATICS 0       /* SingleTrackKinematics  */
#define T2D_MODEL_DYNAMICS 1         /* SingleTrackDynamics    */
#define T2D_MODEL_POINTMASS_NEWTON 2 /* PointMass(backend="newton") */
#define T2D_MODEL_POINTMASS_EULER 3  /* PointMass(backend="euler")  */
#define T2D_MODEL_STATIC 4           /* no motion (Obstacle, obstacle.py:14-19) */
#define T2D_MODEL_DRIFT 5            /* SingleTrackDrift (built-in tyre); needs t2d_bind_wheel_state */

/* collision shape ids (t2d_type_params.shape) */
#define T2D_SHAPE_OBB 0    /* Vehicle / Cyclist / Other bounding box, vehicle.py:132-142 */
#define T2D_SHAPE_CIRCLE 1 /* Pedestrian ((x, y), width/2), pedestrian.py:85-88 */
#define T2D_SHAPE_NONE 2   /* takes part in physics only */

#define T2D_TYPE_INACTIVE 255 /* type id of an empty participant slot */
#define T2D_MAX_TYPES 64
#define T2D_MAX_PARTICIPANTS 128 /* per scenario (one warp spans a scenario) */
#define T2D_MAX_SEGMENTS 32767   /* hit_segment is int16 */
#define T2D_MAX_RANKS 16         /* GPUs of one node sharing a done exchange */
#define T2D_IPC_HANDLE_BYTES 64  /* sizeof(cudaIpcMemHandle_t) */

/* per-participant event byte (t2d_step `flags`) */
#define T2D_F_DYNAMIC 1  /* TrafficStatus.COLLISION_DYNAMIC, status.py:55 */
#define T2D_F_STATIC 2   /* TrafficStatus.COLLISION_STATIC,  status.py:54 */
#define T2D_F_OUTBOUND 4 /* ScenarioStatus.OUT_BOUND,        status.py:26 */

/* scenario status byte = ScenarioStatus, tactics2d/traffic/status.py:23-28 */
#define T2D_STATUS_NORMAL 1
#define T2D_STATUS_COMPLETED 2
#define T2D_STATUS_TIME_EXCEEDED 3
#define T2D_STATUS_OUT_BOUND 4
#define T2D_STATUS_NO_ACTION 5
#define T2D_STATUS_FAILED 6

/* t2d_config.flags */
#define T2D_CFG_ANY_PARTICIPANT 1 /* any active participant's event ends the scenario (default: only participant 0, the ego) */
#define T2D_CFG_STEER_FIRST 2     /* action[...,0] is steering, [...,1] acceleration (env order, parking.py:239) */

typedef struct t2d_ctx t2d_ctx;

typedef struct t2d_config {
  int32_t interval_ms; /* State.frame advance per step; ScenarioManager.step_size (scenario_manager.py:50) */
  int32_t delta_t_ms;  /* Euler sub-step; PhysicsModelBase._DELTA_T = 5 (physics_model_base.py:23) */
  int32_t max_step;    /* TimeExceed.max_step; <= 0 disables the check */
  int32_t flags;       /* T2D_CFG_* */
} t2d_config;

/* One row per participant type.  Ranges are [lo, hi]; "no constraint" (the reference's
 * None) is (-INFINITY, +INFINITY). */
typedef struct t2d_type_params {
  float half_len, half_wid; /* OBB half extents (length/2, width/2) */
  float radius;             /* circle radius (width/2) */
  float lf, lr;             /* axle distances from the geometry centre */
  float steer_lo, steer_hi;
  float speed_lo, speed_hi;
  float accel_lo, accel_hi;
  float mass, mass_height, mu, I_z, cf, cr; /* SingleTrackDynamics only */
  int32_t model;                            /* T2D_MODEL_* */
  int32_t shape;                            /* T2D_SHAPE_* */
  float wheel_radius, T_sb, T_se, I_yw;     /* SingleTrackDrift only (single_track_drift.py:98-107: 0.344, 0.76, 1, 1.7);
                                               the drift model also reads lf, lr, mass, I_z and the three ranges */
} t2d_type_params;

int t2d_version(void);
const char* t2d_last_error(void);

int t2d_create(t2d_ctx** out, int device, int n_scenarios, int m_participants, const t2d_config* cfg);
int t2d_destroy(t2d_ctx* ctx);
int t2d_set_config(t2d_ctx* ctx, const t2d_config* cfg);

/* HOST pointers; copied. */
int t2d_set_type_table(t2d_ctx* ctx, const t2d_type_params* table, int n_types);
/* segments: host float[n_seg][4] = (x1, y1, x2, y2), collidable map polyline pieces in list
 * order (the order defines "first hit"); bounds: host float[4] = (xmin, xmax, ymin, ymax) as
 * Map.boundary gives it, or NULL for no out-of-bound check; cell_size: broadphase grid pitch
 * in metres (<= 0: choose automatically). */
int t2d_set_map(t2d_ctx* ctx, const float* segments, int n_seg, const float* bounds, float cell_size);

/* Static objects that are AREAS, and a different map per scenario.
 * StaticCollision.update tests `agent_pose.intersects(static_object.geometry)` against a list of static objects
 * (traffic/event_detection/collision.py:37-43); in the reference's envs those are Area polygons - the walls and obstacles
 * of a parking lot, regenerated by every reset (envs/parking.py:397-441) - and a pose wholly inside a polygon intersects
 * it without touching an edge.  poly_start (host int32 [n_poly + 1], ascending) marks the segments that close up to
 * rings: ring p = segments [poly_start[p], poly_start[p + 1]), each edge ending where the next begins and the last at the
 * first one's start (Area.geometry's exterior); segments outside every ring are open polyline pieces (RoadLine).
 * With rings present, hit_segment names the first OBJECT hit in list order by its first segment: poly_start[p] for ring p
 * (an edge of it was touched, or the pose centre lies inside it), the segment itself for an open piece. */
int t2d_set_map_polygons(t2d_ctx* ctx, const float* segments, int n_seg, const int32_t* poly_start, int n_poly,
                         const float* bounds, float cell_size);
/* One tile = the static objects + boundary of one map (host arrays, copied).  tile_id: DEVICE uint16 [N], owned by the
 * caller and read by every tick: the tile of each scenario (may be rewritten between ticks, e.g. by a reset that draws a
 * new parking lot); NULL is allowed when n_tiles == 1.  Every scenario then collides with its own tile's objects, is
 * bounded by its own tile's box, and t2d_lidar_scan sees its own tile's segments.
 * A call that is rejected (any T2D_E_INVALID) changes nothing: the previous map stays in force, and with it the previous
 * tile_id array, which the caller must keep alive until a later call succeeds. */
#define T2D_MAX_TILES 4096
typedef struct {
  const float* segments;     /* [n_seg][4] */
  int32_t n_seg;
  const int32_t* poly_start; /* [n_poly + 1] or NULL */
  int32_t n_poly;
  const float* bounds;       /* [4] xmin, xmax, ymin, ymax or NULL */
} t2d_map_tile;
int t2d_set_map_table(t2d_ctx* ctx, const t2d_map_tile* tiles, int n_tiles, const uint16_t* tile_id, float cell_size);

/* DEVICE pointers, each [N, M] (step_count: [N]); read and written in place by t2d_step. */
int t2d_bind_state(t2d_ctx* ctx, float* x, float* y, float* heading, float* speed, float* vx, float* vy,
                   const uint8_t* type_id, int32_t* step_count);

/* SingleTrackDrift carries two more state variables per participant, the front / rear wheel angular speeds that
 * SingleTrackDrift.step takes and returns (single_track_drift.py:467-499).  DEVICE pointers [N, M], read and written in
 * place by t2d_step for participants whose type has model T2D_MODEL_DRIFT; required only when the type table holds
 * such a row. */
int t2d_bind_wheel_state(t2d_ctx* ctx, float* omega_front, float* omega_rear);

/* One tick of all N scenarios.  action: [N, M, 2] fp32.  Outputs (any may be NULL):
 * flags [N, M] uint8, hit_index [N, M] int16 (lowest colliding participant or -1),
 * hit_segment [N, M] int16 (lowest colliding map segment or -1), scn_status [N] uint8,
 * done [N] uint8. */
int t2d_step(t2d_ctx* ctx, const float* action, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment,
             uint8_t* scn_status, uint8_t* done, void* stream);

/* The same tick for a caller whose buffers live in HOST memory - what a ctypes / numpy binding of the reference's
 * env.step(action) -> (..., terminated, truncated, info["status"]) would hand over (envs/parking.py:444-468).
 * action_host: [N, M, 2] fp32 (pinned memory recommended), scn_status_host / done_host: [N] uint8 in host memory
 * (either may be NULL); flags / hit_index / hit_segment stay DEVICE arrays as in t2d_step (any may be NULL).
 * The library stages the actions in chunks of whole scenarios on its own copy stream so that the host->device copy of
 * one chunk runs under the kernel of the previous one, reads status + done back in one device->host copy and
 * synchronises `stream` before returning: the host arrays are valid on return. */
int t2d_step_host(t2d_ctx* ctx, const float* action_host, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment,
                  uint8_t* scn_status_host, uint8_t* done_host, void* stream);

/* The detectors alone on the bound poses (x, y, heading); no physics, no step counting. */
int t2d_check_events(t2d_ctx* ctx, uint8_t* flags, int16_t* hit_index, int16_t* hit_segment, void* stream);

/* Arrival (tactics2d/traffic/event_detection/arrival.py:32-47) and NoAction (no_action.py:32-53) for the ego
 * (participant 0) of every scenario, evaluated inside t2d_step.  All pointers are DEVICE arrays owned by the caller:
 * target [N][5] = (cx, cy, heading, half_len, half_wid) of the target-area rectangle (NULL disables both detectors),
 * iou_out [N] receives IoU(ego pose, target) (Arrival.update's second return value), last_pose [N][4] and
 * no_action_count [N] are the detector state (zero them before the first step; t2d_reset clears them).
 * arrival_threshold: IoU >= threshold -> T2D_STATUS_COMPLETED (reference 0.95); no_action_max_step: more than that
 * many consecutive ticks with IoU(pose, previous pose) > 0.999 -> T2D_STATUS_NO_ACTION (reference 100; <= 0 disables).
 * Status priority (envs/parking.py:361-392): time exceeded, no action, out of bound, collision, completed. */
int t2d_set_goal(t2d_ctx* ctx, const float* target, float arrival_threshold, int no_action_max_step, float* iou_out,
                 float* last_pose, int32_t* no_action_count);

/* Masked re-initialisation (ScenarioManager.reset, envs/parking.py:397-441; ParticipantBase.reset): for every scenario n
 * with mask[n] != 0 copy row pool_index[n] (row n when pool_index is NULL) of the [n_pool, M] pool arrays into the bound
 * state and zero step_count[n]; pool_vx / pool_vy may be NULL (then speed x (cos, sin)(heading)).  Everything else the
 * world owns per participant starts fresh too: the NoAction detector state of t2d_set_goal, the controllers' last_accel
 * (0), and the SingleTrackDrift wheel speeds bound with t2d_bind_wheel_state - from the pool columns of
 * t2d_bind_reset_wheel_pool when bound, else free rolling (speed / wheel_radius). */
int t2d_reset(t2d_ctx* ctx, const uint8_t* mask, const int32_t* pool_index, int n_pool, const float* pool_x,
              const float* pool_y, const float* pool_heading, const float* pool_speed, const float* pool_vx,
              const float* pool_vy, void* stream);
/* Optional initial wheel speeds for t2d_reset: DEVICE arrays [n_pool][M] indexed like the other pool columns (NULL, NULL unbinds). */
int t2d_bind_reset_wheel_pool(t2d_ctx* ctx, const float* pool_omega_front, const float* pool_omega_rear);

/* Single-line lidar of the ego (participant 0) of every scenario: SingleLineLidar._scan_obstacles
 * (tactics2d/sensor/lidar.py:128-221).  n_beams = point_density (lidar.py:49), max_range = perception range;
 * beam_cos_sin: DEVICE double [n_beams][2] = (cos, sin) of the beam angles linspace(0, 2 pi, n_beams, endpoint=False)
 * (lidar.py:160); scan: DEVICE float [N][n_beams], +inf where nothing is hit within the range.  Obstacles are the map
 * segments given to t2d_set_map and the pose rings of the other box-shaped participants. */
int t2d_lidar_scan(t2d_ctx* ctx, int n_beams, float max_range, const double* beam_cos_sin, float* scan, void* stream);

/* On-device NPC controllers (tactics2d/controller).  A controller row is one configured controller object; the fields
 * are the reference's attribute names.  kind selects the law:
 *   T2D_CTRL_IDM           IDMController.step               (steering 0; free flow, or car following when a leader is set)
 *   T2D_CTRL_CRUISE        AccelerationController.step      (steering 0; cruise, or adaptive cruise with a leader)
 *   T2D_CTRL_PURE_PURSUIT  PurePursuitController.step       (pure-pursuit steering on a path + the cruise laws) */
#define T2D_CTRL_EXTERNAL 0 /* the caller's action is kept */
#define T2D_CTRL_IDM 1
#define T2D_CTRL_CRUISE 2
#define T2D_CTRL_PURE_PURSUIT 3
#define T2D_MAX_CONTROLLERS 64

typedef struct t2d_controller_params {
  int32_t kind; /* T2D_CTRL_* */
  /* IDMController.__init__, idm_controller.py:33-58 */
  float desired_speed, time_headway, min_spacing, max_acceleration, comfortable_deceleration, delta;
  /* AccelerationController attributes, acceleration_controller.py:33-39 (after update_driving_style, :62-80) */
  float target_speed, kp, accel_change_rate, delta_t, max_accel, min_accel, interval;
  /* PurePursuitController: min_pre_aiming_distance, interval (pure_pursuit_controller.py:26-36), wheel_base (:76) */
  float min_pre_aiming_distance, pp_interval, wheel_base;
} t2d_controller_params;

/* table: HOST array of n_rows (<= T2D_MAX_CONTROLLERS) rows, copied.  The rest are DEVICE arrays owned by the caller:
 * ctrl_id [N, M] uint8 = row of the participant's controller (255, or a row of kind EXTERNAL: not controlled);
 * lead_index [N, M] int16 = the participant's leading vehicle inside its scenario (`leading_state` / `front_state`),
 * -1 for none (NULL: nobody has one); path_id [N, M] int16 = the pure-pursuit path, -1 for none (NULL allowed);
 * last_accel [N, M] float = |acceleration| each participant applied on the previous tick (State.accel,
 * participant/trajectory/state.py:171-185), read and rewritten by t2d_control; zero it before the first tick.
 * table == NULL removes the controllers. */
int t2d_set_controllers(t2d_ctx* ctx, const t2d_controller_params* table, int n_rows, const uint8_t* ctrl_id,
                        const int16_t* lead_index, const int16_t* path_id, float* last_accel);

/* Pure-pursuit paths: HOST arrays, copied.  xy [V][2] vertices of all paths back to back, offsets [n_paths + 1] (path p
 * owns vertices offsets[p] .. offsets[p + 1] - 1, at least 2). */
int t2d_set_paths(t2d_ctx* ctx, const float* xy, const int32_t* offsets, int n_paths);

/* Overwrites action[n][m] = (accel, steer) ((steer, accel) with T2D_CFG_STEER_FIRST) of every controlled participant from
 * the bound state, then stores |applied acceleration| of the WHOLE action buffer in last_accel (bicycles: the accel clipped
 * to the type's range; point masses: |(ax, ay)|).  Call it after the external actions are in the buffer and before
 * t2d_step.  action: DEVICE [N, M, 2] fp32. */
int t2d_control(t2d_ctx* ctx, float* action, void* stream);

/* ---- the env layer: ego action, host-resident ego caller, reward / terminated / truncated ------------------------------
 * ParkingEnv.step takes ONE action, the ego's (steering, accel) (envs/parking.py:219-239); the other participants of a
 * batched scenario are driven on the device (t2d_control) or by the rows of the caller's action array.
 * t2d_set_ego_action binds a DEVICE array [N][2] (or NULL to unbind): while bound, t2d_control and t2d_step take the
 * action of participant 0 of every scenario from it (t2d_control also writes it into row 0 of `action`). */
int t2d_set_ego_action(t2d_ctx* ctx, const float* ego_action /* device [N][2], 8-byte aligned */);
/* One tick for a caller whose policy lives on the host and drives only the ego: stages ego_action_host [N][2] in pinned,
 * device-mapped host memory that the first kernel reads directly (8 N bytes over PCIe instead of the 8 N M of
 * t2d_step_host, and no copy-engine transfer in front of the kernels), runs t2d_control when controllers are set (the other
 * participants' rows of `action`, a DEVICE array [N][M][2] owned by the caller, never leave the device), the tick, and
 * copies status + done back ([N] each, HOST); synchronises `stream` before returning. */
int t2d_step_host_ego(t2d_ctx* ctx, const float* ego_action_host, float* action, uint8_t* flags, int16_t* hit_index,
                      int16_t* hit_segment, uint8_t* scn_status_host, uint8_t* done_host, void* stream);
/* What ParkingEnv.step computes after check_status (envs/parking.py:240-256, _get_reward :148-190), for all scenarios in
 * one launch, from the tick's outputs `flags` [N][M] and `scn_status` [N]: traffic_status [N][M] (TrafficStatus codes,
 * status.py:52-61; may be NULL), terminated / truncated / done [N] (may be NULL), reward [N] by the reference's chain
 * (-5 collision, -1 time exceeded / no action, -5 out of bound, +5 completed, else time penalty + IoU gain + 0.1 x
 * progress towards the target).  max_iou / min_dist [N]: the per-episode extrema the reward keeps (ParkingEnv._max_iou,
 * _min_dist_to_target; initialise to -inf / +inf; NULL when no goal is set); with reset_trackers_on_done they are
 * re-initialised for the scenarios that are done, so that `done` can go straight into t2d_reset.  All arrays DEVICE. */
int t2d_env_epilogue(t2d_ctx* ctx, const uint8_t* flags, const uint8_t* scn_status, float* reward, uint8_t* terminated,
                     uint8_t* truncated, uint8_t* traffic_status, uint8_t* done, float* max_iou, float* min_dist,
                     int reset_trackers_on_done, void* stream);

/* ---- done-mask exchange across the GPUs of one node, over peer memory (NVLink / NVSwitch) -------------------------
 * Scenarios are sharded across ranks (one process per GPU); the one exchange of the path is "every rank learns every
 * rank's done mask of this tick" - the terminated / truncated vector a central learner or reset scheduler reads
 * (envs/parking.py:243-248 per scenario).  t2d_exchange_allgather is that all-gather as ONE small kernel per rank:
 * it stores the rank's mask into a ring slot on EVERY rank (peer stores), signals the step on every rank's flag word
 * (release, system scope), waits for all ranks' signals of the same step (acquire; bounded - a rank that never shows
 * up sets the sticky timed_out word instead of hanging the GPU) and copies the slot to the caller's array.
 *
 * Set-up: every rank calls t2d_exchange_create (fills a 64-byte CUDA IPC handle), the ranks pass the handles around
 * by any host channel (torch.distributed in this repository), every rank calls t2d_exchange_connect with all `world`
 * handles in rank order.  n_local = scenarios per rank (rows are padded to a multiple of 16); slots >= 2 = ring depth.
 * Every rank must call t2d_exchange_allgather the same number of times, in stream order on each rank. */
typedef struct t2d_exchange t2d_exchange;
int t2d_exchange_create(t2d_exchange** out, int device, int world, int rank, int n_local, int slots, void* ipc_handle_out);
int t2d_exchange_connect(t2d_exchange* x, const void* handles /* host, world x T2D_IPC_HANDLE_BYTES */);
/* done_local: DEVICE uint8 [n_local] (t2d_step's `done`); dst: DEVICE uint8 [world * ((n_local + 15) & ~15)], rank order. */
int t2d_exchange_allgather(t2d_exchange* x, const uint8_t* done_local, uint8_t* dst, void* stream);
/* The same exchange taken off the critical path: the call posts this step's mask (put + signal, nothing to wait for)
 * and delivers into dst the gathered masks of the step `lag` calls earlier, whose signals have long arrived (the first
 * `lag` calls deliver nothing and leave dst untouched).  The consumer of the gathered masks - a central learner or
 * reset scheduler - is behind the simulation anyway; the ticks of the ranks no longer meet once per step.
 * Needs slots >= 2 * lag + 2.  lag = 0 is t2d_exchange_allgather.  If a rank fails to signal within the time-out
 * (T2D_EXCHANGE_TIMEOUT_MS, default ~2 s) dst is filled with 0xFF and the sticky timed_out word is set. */
int t2d_exchange_allgather_lagged(t2d_exchange* x, const uint8_t* done_local, uint8_t* dst, int lag, void* stream);
int t2d_exchange_status(t2d_exchange* x, uint32_t* steps, uint32_t* timed_out);
int t2d_exchange_destroy(t2d_exchange* x);

/* Flat batch of `n` independent participants through ONE model (PhysicsModelBase.step):
 * state arrays are read and written in place; action [n, 2]; applied [n, 2] (may be NULL)
 * receives the clipped (accel, steer) the reference returns next to the State.  omega_front / omega_rear [n]: the wheel
 * speeds of SingleTrackDrift.step (in / out); NULL for every other model. */
int t2d_physics_step(int device, const t2d_type_params* params /*host*/, int interval_ms, int delta_t_ms, int n,
                     float* x, float* y, float* heading, float* speed, float* vx, float* vy, float* omega_front,
                     float* omega_rear, const float* action, float* applied, void* stream);

/* Diagnostics: device buffer int64[ceil(N / scenarios_per_warp)][10] that receives clock64() at the eight phase
 * boundaries of every warp tile of t2d_step (load, physics, pose, pair loop, pair drain, static, out-of-bound, end), the SM id and the warp's kernel-entry clock;
 * NULL (default) disables it.  Used by profiles/phase_clocks.py. */
int t2d_debug_set_clock_buffer(t2d_ctx* ctx, long long* device_buffer);

/* Tuning knob of t2d_step, no effect on results: the tick can ask L2 for its first input lines while the previous grid is
 * still draining (and for the next tile inside its persistent loop).  mode 1: on, 0: off, -1 (default): on unless a
 * peer-memory done exchange is alive in the process (on one GPU it saves ~1 us per tick at 4096 x 64; next to the
 * exchange kernel on 8 GPUs it measured slower).  A caller that can time both settings picks with this (bench.py does at
 * N > 1); the environment variable T2D_PREFETCH sets the initial mode at t2d_create. */
int t2d_set_prefetch(t2d_ctx* ctx, int mode);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t t2d_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* T2D_B200_H */
