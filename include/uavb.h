/*
 * uavb.h -- C ABI of the B200-native batched closed-loop flight path (libuavb.so).
 *
 * The reference (Mdhvince/UAV-Autonomous-control) is pure Python and has no FFI; the seams this
 * library replaces are plain Python calls between objects (SURVEY.md 8(b)).  Every entry point
 * below names the reference interface it stands in for (paths relative to /root/reference).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++ or torch types.
 *   - return 0 on success, a negative UAVB_E* code otherwise; uavb_last_error() returns a
 *     thread-local message for the last failing call on this thread.
 *   - unless the name ends in _host, every pointer is a DEVICE pointer owned by the caller, the
 *     work is enqueued on `stream` (a cudaStream_t passed as void*, NULL = default stream) and the
 *     call returns without synchronising.  No hidden global state: calls on different streams or
 *     threads do not interact.
 *   - *_host entry points take HOST pointers, copy host->device, launch, copy device->host and
 *     synchronise before returning (the end-to-end path a ctypes / cgo style binding would use).
 *   - there is NO CPU implementation behind this ABI: on a machine without a CUDA device every
 *     compute entry point fails with UAVB_ENODEVICE.
 *   - frames: NED world / FRD body, scalar-first quaternion, state X = [x y z  q0 q1 q2 q3
 *     vx vy vz  p q r] exactly as uav_ac/quadrotor/quad.py:75-80.
 */
#ifndef UAVB_H
#define UAVB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UAVB_VERSION 210            /* 0.2.1: uavb_minsnap_correct_f64 / uavb_minsnap_pack_f64, uavb_mission_host.plan_aabbs / no_correction (0.2.0: two drones per thread, packed fp32x2 tick, uavb_rollout_args.n_slices) */

#define UAVB_OK          0
#define UAVB_EINVAL     -1          /* bad argument (null pointer, size out of range) */
#define UAVB_ECUDA      -2          /* CUDA runtime error, see uavb_last_error() */
#define UAVB_ENODEVICE  -3          /* no CUDA device / wrong architecture */
#define UAVB_ENOMEM     -4

#define UAVB_N_COEFFS    8          /* coefficients per spline and axis: minimum_snap.py:28 */
#define UAVB_STATE_DIM  13          /* quad.py:75-80 */
#define UAVB_N_GAINS    11          /* kp_xy kd_xy kp_z kd_z ki_z kp_roll kp_pitch kp_yaw kp_p kp_q kp_r (quad.py:65-73) */
#define UAVB_N_METRICS   8
#define UAVB_CARRY_WORDS 52         /* 32-bit words per rollout in the resumable carry block */
#define UAVB_MAX_SPLINES 64         /* upper bound on splines per mission accepted by the solver */

/* per-mission solver status (status_out of uavb_minsnap_solve_f64) */
#define UAVB_SOLVE_OK        0
#define UAVB_SOLVE_DEGENERATE 1     /* a segment has zero length (T_i = 0) or velocity <= 0: KKT singular
                                       (np.linalg.solve would raise LinAlgError, minimum_snap.py:151) */
#define UAVB_SOLVE_NONFINITE 2      /* non-finite input or result */
#define UAVB_SOLVE_TOO_MANY  3      /* more splines than the caller's capacity / UAVB_MAX_SPLINES (the correction loop kept
                                       inserting midpoints: an obstacle probably contains a waypoint -- the reference loops forever) */

/* per-rollout status bits (metrics column 5 and status_out of uavb_rollout_f32) */
#define UAVB_ROLLOUT_OK        0
#define UAVB_ROLLOUT_NONFINITE 1    /* state became NaN/Inf (the reference has no guard: controller.py:50,150,167) */
#define UAVB_ROLLOUT_DIVERGED  2    /* tracking error exceeded 1e4 m */

/* metrics_out columns */
#define UAVB_M_FINAL_DIST 0         /* |p - goal| after the last tick            (main.py:115)            */
#define UAVB_M_COLLISION  1         /* 1.0 if the body origin was ever inside an AABB (minimum_snap.py:327-357) */
#define UAVB_M_RMSE       2         /* sqrt(mean e^2), e = per-outer-period tracking error                */
#define UAVB_M_MEAN_ERR   3         /* mean e (tests/integration/test_mujoco_trajectory_tracking.py:31,35) */
#define UAVB_M_MAX_ERR    4
#define UAVB_M_STATUS     5         /* UAVB_ROLLOUT_* bits as a float                                     */
#define UAVB_M_FIRST_HIT  6         /* tick index of the first AABB hit, -1 if none                       */
#define UAVB_M_PERIODS    7         /* number of outer periods that contributed to the error statistics  */

int         uavb_version(void);
const char* uavb_last_error(void);
/* Number of visible CUDA devices (0 on a GPU-less host; never fails). */
int         uavb_device_count(void);
/* SM count and compute capability of device `dev`; UAVB_ENODEVICE without a GPU. */
int         uavb_device_info(int dev, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------------
 * K1  minimum-snap solve, fp64, one thread per mission.
 *
 * Replaces MinimumSnap._compute_spline_parameters (uav_ac/planning/minimum_snap.py:138-153) together
 * with _generate_time_per_spline (:311-321) for B missions at once.  The unique solution of the
 * reference's KKT system [[Q,A^T],[A,0]] (rows listed at :171-255, Q at :155-169) is computed from
 * its reduced form: the free unknowns are velocity/acceleration/jerk at the S-1 interior waypoints,
 * the stationarity conditions form an SPD block-tridiagonal system with 3x3 blocks that is solved
 * in registers (block Thomas elimination, LDL^T blocks), and the 8 coefficients of every spline follow in closed form (DESIGN.md "K1").
 *
 *   waypoints  [B][S+1][3]  row-major, NED metres
 *   velocity   [B]          cruise speed of each mission (minimum_snap.py:13 `velocity`)
 *   start_end_time_factor   MinimumSnap.START_END_TIME_FACTOR (1.5, minimum_snap.py:10)
 *   coeffs_out [B][8*S][3]  row 8*i+j = coefficient of t^j of spline i -- the layout of the
 *                           reference attribute MinimumSnap.coeffs (minimum_snap.py:153)
 *   times_out  [B][S]       MinimumSnap.times
 *   status_out [B]          UAVB_SOLVE_*; may be NULL
 * 1 <= S <= UAVB_MAX_SPLINES.
 */
int uavb_minsnap_solve_f64(const double* waypoints, const double* velocity, int B, int S,
                           double start_end_time_factor, double* coeffs_out, double* times_out,
                           int* status_out, void* stream);

/* Ragged variant: mission b owns waypoints [wp_offsets[b], wp_offsets[b+1]) of the packed array and
 * S_b = wp_offsets[b+1]-wp_offsets[b]-1 splines; its first spline is packed segment
 * wp_offsets[b]-b.  coeffs_out [n_seg][8][3], times_out [n_seg], n_seg = wp_offsets[B]-B.
 * Used by the obstacle-correction loop (minimum_snap.py:63-95) where midpoint insertion makes S
 * differ between missions. */
int uavb_minsnap_solve_ragged_f64(const double* waypoints, const int* wp_offsets, const double* velocity,
                                  int B, double start_end_time_factor, double* coeffs_out,
                                  double* times_out, int* status_out, void* stream);

/* The reference's constraint system, MinimumSnap.A and MinimumSnap.b after _create_polynom_matrices (minimum_snap.py:171-255),
 * in the reference's row order: 2S position rows, 6 boundary rows, 4 (S-1) continuity rows.  K1 does not use it (it solves the
 * reduced problem); it serves the attribute surface of the reference class and its KKT-optimality test
 * (tests/unit/planning/test_minimum_snap.py:154-168).
 *   waypoints [B][S+1][3], times [B][S] (MinimumSnap.times)  ->  A_out [B][6S+2][8S], b_out [B][6S+2][3] */
int uavb_minsnap_constraints_f64(const double* waypoints, const double* times, int B, int S, double* A_out, double* b_out,
                                 void* stream);

/* Table geometry of MinimumSnap._generate_trajectory (minimum_snap.py:97-124) without sampling it:
 *   rows_out  [n_seg]  len(np.arange(0, T_i, dt)) of every packed segment (:104)
 *   yaw0_out  [B]      yaw taken by the rows that precede the first row with horizontal speed
 *                      >= 1e-3 (the look-ahead of _calculate_yaws, :126-136); 0 when no row is valid
 *   total_rows_out [B] rows of the whole table of mission b; may be NULL
 * seg_offsets [B+1] gives the packed segment range of every mission. */
int uavb_minsnap_table_meta_f64(const double* coeffs, const double* times, const int* seg_offsets, int B,
                                double dt, int* rows_out, double* yaw0_out, int* total_rows_out, void* stream);

/* K3  sampled table, the (N, 11) array returned by MinimumSnap.get_trajectory()
 * (minimum_snap.py:59-61, 97-124): [x y z  vx vy vz  ax ay az  yaw  spline_id].
 *   row_offsets [B+1]  exclusive prefix sum of total rows per mission (from uavb_minsnap_table_meta_f64)
 *   table_out   [row_offsets[B]][11]
 * Yaw uses hold-last-valid and np.unwrap semantics per mission (:126-136). */
int uavb_minsnap_sample_f64(const double* coeffs, const double* times, const int* seg_offsets,
                            const int* seg_rows, const int* row_offsets, int B, double dt,
                            double* table_out, void* stream);

/* MinimumSnap._calculate_yaws (minimum_snap.py:126-136) on bare velocity rows: heading of the horizontal velocity where
 * its norm reaches 1e-3, np.unwrap over the valid rows, hold-last-valid, first-valid look-ahead, zeros if none is
 * valid.  velocities [n_rows][3]; sequence b owns rows [row_offsets[b], row_offsets[b+1]); yaws_out [n_rows]. */
int uavb_minsnap_yaw_profile_f64(const double* velocities, const int* row_offsets, int B, long long n_rows,
                                 double* yaws_out, void* stream);

/* Inclusive point-in-AABB over sampled tables, the test of the correction loop
 * (minimum_snap.py:84-87 with is_collision_cuboid :327-357).  For every mission b, ORs into
 * hit_mask_out[b] (uint64, bit s) the splines s that have a sampled row inside `cuboid` (6 doubles,
 * [xmin xmax ymin ymax zmin zmax]).  cuboid_stride = 0: one cuboid for all missions, 6: one each. */
int uavb_minsnap_table_hits_f64(const double* table, const int* row_offsets, int B, const double* cuboid,
                                int cuboid_stride, unsigned long long* hit_mask_out, void* stream);

/* The obstacle-correction loop of MinimumSnap._generate_collision_free_trajectory (minimum_snap.py:63-95) for B missions,
 * entirely on the device: for every obstacle in order, plan (K1), find the splines that own a sampled row (j * dt,
 * j < len(np.arange(0, T_i, dt)), :104) inside the box (is_collision_cuboid, :327-357), insert the midpoint of each as a new
 * waypoint (insert_midpoints_at_indexes, :359-391) and plan again until the table is clean.  Every mission walks the obstacle
 * list with its own cursor; only missions that were hit are planned again (DESIGN.md "correction loop").
 *   waypoints    [B][max_wp][3]  in/out, fixed pitch: mission b uses rows [0, n_waypoints[b])
 *   n_waypoints  [B]             in/out
 *   cuboids      [n_obs][6] doubles [xmin xmax ymin ymax zmin zmax] shared by all missions (cuboid_stride 0), or one set per
 *                mission, cuboid_stride doubles apart;  n_obs = 0 plans without obstacles
 *   coeffs_out   [B][max_wp-1][8][3], times_out [B][max_wp-1]  fixed pitch, the first n_waypoints[b]-1 splines are valid
 *   status_out   [B] UAVB_SOLVE_* (required); UAVB_SOLVE_TOO_MANY when a mission would need more than max_wp waypoints
 *   rounds_out   HOST int, plan rounds run (1 = nothing was hit); may be NULL
 * max_wp <= UAVB_MAX_SPLINES + 1.  Unlike the other device-pointer entry points this one SYNCHRONISES `stream` (the host reads
 * four counters per round to size the next one). */
int uavb_minsnap_correct_f64(double* waypoints, int* n_waypoints, const double* velocity, int B, int max_wp,
                             double start_end_time_factor, double dt, const double* cuboids, int n_obs, long long cuboid_stride,
                             double* coeffs_out, double* times_out, int* status_out, int* rounds_out, void* stream);

/* Fixed pitch -> packed segments: spline s of mission b (s < n_waypoints[b]-1) goes to packed segment seg_offsets[b] + s.
 * seg_offsets [B] (or [B+1]) = exclusive prefix sum of n_waypoints-1, provided by the caller. */
int uavb_minsnap_pack_f64(const double* coeffs, const double* times, const int* n_waypoints, int B, int max_wp,
                          const int* seg_offsets, double* coeffs_out, double* times_out, void* stream);

/* One mission made of n_tables consecutive MinimumSnap tables -- _generate_mission_trajectory's vertical take-off + course
 * (main.py:73-84) -- each planned with the correction loop above, laid out as the packed segment arrays of a shared-mission
 * rollout (struct uavb_rollout_args).  ONE host synchronisation when nothing is hit (the usual case).
 *   table_waypoints    HOST array of n_tables DEVICE pointers, table k = [table_n_waypoints[k]][3] doubles
 *   table_n_waypoints  HOST array [n_tables];   table_velocity  DEVICE array [n_tables]
 *   cuboids            DEVICE [n_obs][6] doubles, n_obs = 0 plans the waypoints as given
 *   seg_coeffs [cap_seg][8][3], seg_times / seg_rows / seg_table / seg_yaw0 [cap_seg]   DEVICE outputs; cap_seg >= the splines
 *                      of the corrected mission (n_tables * UAVB_MAX_SPLINES always suffices)
 *   n_seg_out, rows_out [n_tables] (table rows of every table), status_out [n_tables] (UAVB_SOLVE_*), rounds_out (may be NULL)  HOST
 * SYNCHRONISES `stream`, n_tables <= 8 -- unless async_report is given.
 *
 * async_report (PINNED host memory, UAVB_PLAN_REPORT_INTS ints, or NULL): the SPECULATIVE form for a caller that plans the same
 * mission again and again (a Monte-Carlo job) and does not want a host round trip per plan.  The call enqueues the plan as it is
 * when nothing is hit and returns at once (n_seg_out = the uncorrected spline count, rows_out / status_out untouched); `stream`
 * later delivers the loop's control block into async_report.  After synchronising with that copy the caller MUST check it:
 *   async_report[4..7] all zero  (no mission was hit: the plan stands),
 *   async_report[8 + n_tables + k] == UAVB_SOLVE_OK and async_report[8 + 2 n_tables + k] = table rows of table k.
 * If a counter is non-zero the segment arrays hold the plan BEFORE correction: plan again without async_report. */
#define UAVB_PLAN_REPORT_INTS 128     /* the first half is the report, the second half the call's upload image */
int uavb_plan_shared_f64(int n_tables, const double* const* table_waypoints, const int* table_n_waypoints, const double* table_velocity,
                         double start_end_time_factor, double dt, const double* cuboids, int n_obs, int cap_seg, double* seg_coeffs,
                         double* seg_times, int* seg_rows, int* seg_table, double* seg_yaw0, int* n_seg_out, int* rows_out, int* status_out,
                         int* rounds_out, int* async_report, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2  persistent closed-loop rollout, fp32 state in registers, one thread per drone.
 */
typedef struct uavb_vehicle {
  /* Quad.__init__ arguments (uav_ac/quadrotor/quad.py:11-51) and lab_course.xml constants */
  double g, dt;                                   /* gravity, inner (physics) time step             */
  double mass, inertia[3];
  double arm, kf, kappa;                          /* lever arm, force coefficient, drag-to-thrust   */
  double min_thrust, max_thrust;                  /* per rotor                                      */
  double tau_rise, tau_fall;                      /* motor time constants                           */
  double max_ascent, max_descent, max_speed_xy, max_horiz_accel, max_tilt;   /* flight limits       */
  double gains[UAVB_N_GAINS];                     /* order of UAVB_N_GAINS above (quad.py:65-73)    */
  double integral_limit;                          /* CascadedController.INTEGRAL_ERROR_LIMIT (controller.py:10) */
} uavb_vehicle;

typedef struct uavb_rollout_args {
  int B;                      /* rollouts in this launch                                            */
  int n_ticks;                /* inner ticks to advance (every rollout the same number)             */
  int inner_per_outer;        /* config.ini `frequency` (main.py:39): outer loop every N ticks      */
  int thrust_frame_lag;       /* 1 = headless loop (stale data.xmat, SURVEY 3.2), 0 = viewer path   */
  int resume;                 /* 0: initialise from `start`; 1: continue from `carry`               */
  int log_stride;             /* 0 = no state log; else one sample after every log_stride ticks     */
  int n_obs;                  /* AABBs per obstacle set                                              */
  int n_obs_sets;             /* number of obstacle sets in `aabbs` (>= 1 when n_obs > 0)            */
  long long index_base;       /* global index of rollout 0 of this launch (sharding; informational) */

  uavb_vehicle veh;           /* defaults for every rollout                                          */

  /* optional per-rollout Monte-Carlo overrides, SoA, NULL = use veh.* (BASELINE configs[2..3]) */
  const float* mc_mass;       /* [B]                                                                 */
  const float* mc_inertia;    /* [3][B]                                                              */
  const float* mc_gains;      /* [UAVB_N_GAINS][B]                                                   */
  const float* mc_wind;       /* [3][B] constant world-frame force in N (extension, not in reference) */

  /* mission: packed segments in the reference coefficient layout (MinimumSnap.coeffs rows) */
  const double* seg_coeffs;   /* [n_seg][8][3]                                                       */
  const int*    seg_rows;     /* [n_seg] table rows of each segment (uavb_minsnap_table_meta_f64)     */
  const int*    seg_table;    /* [n_seg] 1 where a new MinimumSnap table starts (yaw hold restarts:
                                  main.py:80-84 stitches two independent tables), else 0              */
  const double* seg_yaw0;     /* [n_seg] yaw0 of the table that starts at this segment (else unused)  */
  const int*    mission_seg_begin;  /* [B] first packed segment of each rollout, NULL = 0 for all     */
  const int*    mission_seg_count;  /* [B] segments of each rollout, NULL = n_seg_shared for all      */
  int           n_seg_shared;
  double        dt_outer;     /* table sampling period, quad.dt * frequency (main.py:97)             */
  const void*   shared_targets;   /* optional, shared missions only: the per-row set-points precomputed by
                                     uavb_rollout_targets_f64 ([n_target_rows] records of 56 bytes); NULL = the kernel
                                     evaluates the polynomials itself.  Both forms give bit-identical rollouts.        */
  int           n_target_rows;
  int           n_slices;     /* 0 = library policy (one slice when every work group has a resident CTA, otherwise slices of
                                 decreasing length: each a fifth of the remaining ticks, at least 200).  > 0: cut the launch into
                                 this many EQUAL time slices (fp32 only; clamped to whole outer periods of >= 100 ticks).
                                 Per-rollout results do not depend on it -- the tests fly the same batch with several values to
                                 prove exactly that.                                                                    */

  const double* start;        /* initial position, [3] (start_stride 0) or [B][3] (start_stride 3)    */
  int           start_stride;
  const double* goal;         /* goal for final_dist, same striding; NULL = no final_dist (0)         */
  int           goal_stride;

  const float*  aabbs;        /* [n_obs_sets][n_obs][6] = [xmin xmax ymin ymax zmin zmax]              */
  const int*    aabb_set;     /* [B] obstacle set of each rollout, NULL = set 0                        */

  float*        carry;        /* [UAVB_CARRY_WORDS][B] resumable rollout state (in when resume, always out); may be NULL when resume = 0 */
  float*        state_out;    /* [13][B] final X, SoA; may be NULL                                     */
  float*        metrics_out;  /* [B][UAVB_N_METRICS]; may be NULL                                      */
  float*        log_out;      /* [n_ticks / log_stride][13][B] SoA samples; required iff log_stride > 0 */
  /* D5, the viewer's flown-path list (MujocoSimulation._record_actual_trajectory, mujoco_sim.py:201-218), per rollout: after every
     tick the simulation time advances by veh.dt (mj_step); the position is appended when z <= traj_gate_z (NED: at or above the
     take-off altitude, mission_waypoints[1][2]) and time >= next sample time, which then becomes time + traj_interval.
     fp32 rollouts only; not together with log_out.  Rollout i's k-th sample is traj_out[k][0..2][i]. */
  float*        traj_out;         /* [traj_max_samples][3][B] or NULL                                                     */
  int*          traj_count_out;   /* [B] samples the reference would hold (may exceed traj_max_samples; the rest is dropped) */
  int           traj_max_samples;
  double        traj_gate_z;
  double        traj_interval;    /* ACTUAL_TRAJECTORY_SAMPLE_INTERVAL = 0.05 s (mujoco_sim.py:16)                       */
  /* Optional unilateral floor (SURVEY 7.3: the reference's drone rests on MuJoCo's ground plane until the rotors carry it; a free body
     sags ~1.5 cm through it during the first 50 ms).  ground_on = 1: after every tick, z > ground_z (NED, below the floor) is set
     back to ground_z and a downward velocity to zero.  Default 0: free body, as in round 1. */
  int           ground_on;
  double        ground_z;
  int           pair_kernel_only; /* 0 = library policy: metrics-only fp32 rollouts with per-rollout missions fly one drone per thread
                                     (the round-1 kernel, faster on such divergent batches), everything else two per thread;
                                     1 = always two per thread.  Both meet the 1e-4 budget; their bits differ.                  */
  int           log_tma;      /* 0 = library policy: the fp32 log leaves through staged TMA tensor stores when B is a multiple of 4 and
                                 log_out is 16-byte aligned, else through per-thread streaming stores; -1 = always the latter (same bits) */
} uavb_rollout_args;

/* Set-points of every table row of ONE mission (the rows MinimumSnap._generate_trajectory would sample, :97-124, plus the
 * heading rule of _calculate_yaws as a direction): x y z in fp64, velocity / acceleration / heading direction in fp32,
 * 56 bytes per row.  A shared-mission rollout that receives this table reads one row per outer period instead of
 * evaluating 9 polynomials per drone.  segment arrays as in uavb_rollout_args (n_seg segments of one mission);
 * targets_out holds n_rows = sum(seg_rows) records. */
#define UAVB_TARGET_ROW_BYTES 56
int uavb_rollout_targets_f64(const double* seg_coeffs, const int* seg_rows, const int* seg_table, const double* seg_yaw0,
                             int n_seg, double dt_outer, void* targets_out, int n_rows, void* stream);

/* Execution (DESIGN.md "K2"): fp32 launches fly TWO drones per thread (rollouts 2j and 2j+1 in the two lanes of packed
 * fp32x2 registers) on a persistent grid of 8 one-warp CTAs (64 drones each) per SM at 255 registers; when the
 * batch exceeds that capacity the mission is cut into time slices that CTAs pull from an atomic work queue, a drone
 * resting in the carry block between slices (scratch comes from a library-private stream-ordered pool when `carry` is
 * NULL); a state log is written slice by slice into its place.  One compiled body per mode serves every batch size, so
 * per-rollout results do not depend on B, on index_base or on how a job is sharded over launches and GPUs.  Launches with
 * a state log (log_stride > 0) renormalise the quaternion every tick, metrics-only launches once per outer period
 * (state_out is unit either way).  uavb_rollout_f64 runs one-shot.
 *
 * Replaces, for B drones and n_ticks ticks, the loop
 *     trajectory_controller.step(); simulation.step()
 * of tests/integration/test_mujoco_trajectory_tracking.py:27-31, i.e. TrajectoryController.step
 * (uav_ac/main.py:37-61), CascadedController.{altitude,lateral,reduced_attitude,body_rate_controller}
 * (uav_ac/control/controller.py:26-168), Quad.set_propeller_speed/_allocate_rotor_forces
 * (uav_ac/quadrotor/quad.py:88-122), MujocoSimulation.step (uav_ac/simulation/mujoco_sim.py:144-151,
 * restated as a free rigid body) and the table rows of MinimumSnap._generate_trajectory
 * (minimum_snap.py:97-124) evaluated on the fly. */
int uavb_rollout_f32(const uavb_rollout_args* args, void* stream);

/* Same rollout with every state variable and operation in fp64 (validation of the fp32 path).  Waypoint missions only: caller
 * tables (uavb_rollout_tables_f32) have no fp64 form. */
int uavb_rollout_f64(const uavb_rollout_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Caller-supplied trajectory tables: the seam TrajectoryController(controller, quad, trajectory, frequency) (main.py:10-61)
 * flies ANY (N, 11) table [x y z vx vy vz ax ay az yaw spline_id], one row per outer period, the index clamped at the last row.
 *
 * uavb_table_targets_f64: tables [n_rows][11] fp64 (several tables may be packed one after the other) -> targets_out [n_rows]
 * records of UAVB_TARGET_ROW_BYTES: x y z copied, velocity / acceleration rounded once to fp32, the yaw column (the set-point the
 * reference feeds to yaw_controller, main.py:58) as the heading direction (cos yaw, sin yaw) computed in fp64 -- yaw and
 * yaw + 2 pi k are the same set-point, as in controller.py:156-168.  No hold-last-valid rule is applied (that belongs to table
 * generation, minimum_snap.py:126-136); the spline_id column is ignored; non-finite values pass through (the rollout then reports
 * UAVB_ROLLOUT_NONFINITE). */
int uavb_table_targets_f64(const double* tables, long long n_rows, void* targets_out, void* stream);

typedef struct uavb_table_set {
  const void*      rows;         /* DEVICE [n_rows] UAVB_TARGET_ROW_BYTES records (uavb_table_targets_f64)                          */
  const long long* offsets;      /* DEVICE [n_tables + 1]: table t = rows [offsets[t], offsets[t+1]), >= 1 row each                  */
  const int*       table_index;  /* DEVICE [B] table of every rollout, 0 <= table_index[b] < n_tables; NULL = rollout b flies table b
                                    (n_tables == B)                                                                                    */
  int              n_tables;
  int              shared_rows;  /* > 0: ONE table of this many rows flown by every rollout (offsets / table_index NULL, n_tables unused) */
} uavb_table_set;

/* The fp32 rollout of uavb_rollout_f32 with the set-points read from caller tables: inner_per_outer ticks per table row, the row
 * index clamped at each rollout's own last row (main.py:61).  Every mission-segment field of `args` must be NULL / 0 (seg_*,
 * mission_seg_*, n_seg_shared, shared_targets, n_target_rows), otherwise UAVB_EINVAL; dt_outer is not read (the controller's outer
 * period is veh.dt * inner_per_outer).  Everything else keeps its meaning: Monte-Carlo overrides, obstacle sets, floor, state log,
 * flown-path list, start / goal strides, n_slices, carry / resume (the carry holds the row relative to the rollout's table: resume
 * with the same table set) and index_base.  A shared table runs the shared-mission kernels of uavb_rollout_f32; per-rollout tables
 * run kernels that read one record per lane and outer period.  The table set is not range-checked on the device: offsets must be
 * non-decreasing with >= 1 row per table and table_index inside [0, n_tables). */
int uavb_rollout_tables_f32(const uavb_rollout_args* args, const uavb_table_set* tables, void* stream);

/* Fill `veh` with the lab_course.xml vehicle and the gains of Quad.__init__ (quad.py:54-73). */
void uavb_vehicle_defaults(uavb_vehicle* veh);

/* ------------------------------------------------------------------------------------------------
 * Stage-level entry points: one controller / vehicle method for B drones (unit-test granularity; the
 * batched Python classes CascadedController / Quad / TrajectoryController call these).
 * All arrays fp32 SoA with the drone index fastest; X is [13][B].
 *
 *   stage        replaces                                                  reads                      writes
 *   OUTER        TrajectoryController._update_outer_loop (main.py:47-61)   X target integral          thrust pqr_cmd integral
 *   INNER        body_rate_controller + set_propeller_speed (main.py:42-44) X thrust pqr_cmd omega     moment forces omega omega_cmd
 *   PHYSICS      MujocoSimulation.step (mujoco_sim.py:144-151, free body)  X omega [zb] [wind] [aabbs] X [zb_out] [collided]
 *   ALTITUDE     CascadedController.altitude (controller.py:26-56)         X target[2,5,8] [rot] integral   thrust integral
 *   LATERAL      CascadedController.lateral (controller.py:58-97)          X target[0,1,3,4,6,7] thrust     bxy
 *   ROLL_PITCH   roll_pitch_controller (controller.py:132-154)             bxy, rot or X              pqr_cmd[0..1]
 *   YAW          yaw_controller (controller.py:156-168)                    X target[9] pqr_cmd[1]     pqr_cmd[2]
 *   BODY_RATE    body_rate_controller (controller.py:115-130)              X pqr_cmd                  moment
 *   ALLOCATE     Quad._allocate_rotor_forces (quad.py:105-122)             thrust moment              forces
 *   PROPELLER    Quad.set_propeller_speed (quad.py:88-103)                 thrust moment omega        forces omega omega_cmd
 *   ATTITUDE     Quad.R() and phi/theta/psi (quad.py:129-155, 189-213)     X                          rot euler
 * Arrays a stage does not use may be NULL.  Outputs marked optional in the struct may be NULL as well.
 */
#define UAVB_STAGE_OUTER       1
#define UAVB_STAGE_INNER       2
#define UAVB_STAGE_PHYSICS     3
#define UAVB_STAGE_ALTITUDE    4
#define UAVB_STAGE_LATERAL     5
#define UAVB_STAGE_ROLL_PITCH  6
#define UAVB_STAGE_YAW         7
#define UAVB_STAGE_BODY_RATE   8
#define UAVB_STAGE_ALLOCATE    9
#define UAVB_STAGE_PROPELLER  10
#define UAVB_STAGE_ATTITUDE   11
typedef struct uavb_stage_args {
  int B;
  int stage;
  uavb_vehicle veh;
  double dt_outer;           /* CascadedController.dt (controller.py:18) */
  /* optional per-drone overrides, as in uavb_rollout_args (the reference passes gains as method arguments) */
  const float* mc_mass;      /* [B] */
  const float* mc_inertia;   /* [3][B] */
  const float* mc_gains;     /* [UAVB_N_GAINS][B] */
  const float* wind;         /* [3][B] */
  float* X;                  /* [13][B] */
  const float* target;       /* [10][B]: x y z vx vy vz ax ay az yaw of the table row */
  const float* rot;          /* [9][B] row-major rotation matrix argument of altitude / roll_pitch_controller; NULL = from X */
  float* integral;           /* [B] CascadedController.integral_error */
  float* thrust;             /* [B] */
  float* bxy;                /* [2][B] */
  float* pqr_cmd;            /* [3][B] */
  float* moment;             /* [3][B] (optional output of INNER) */
  float* forces;             /* [4][B] (optional output of INNER / PROPELLER) */
  float* omega;              /* [4][B] Quad.omega */
  float* omega_cmd;          /* [4][B] Quad.omega_command (optional output) */
  const float* zb;           /* [3][B] thrust direction for PHYSICS (third column of the stale body rotation); NULL = from X */
  float* zb_out;             /* [3][B] PHYSICS: body z axis of the state BEFORE the step (the next call's stale thrust frame) */
  const float* aabbs;        /* [n_obs][6] PHYSICS: obstacles for the sticky collision flag (minimum_snap.py:327-357) */
  int n_obs;
  float* collided;           /* [B] PHYSICS: set to 1 when the body origin is inside a box after the step (never cleared) */
  float* rot_out;            /* [9][B] ATTITUDE */
  float* euler_out;          /* [3][B] ATTITUDE: phi theta psi */
} uavb_stage_args;
int uavb_stage_f32(const uavb_stage_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Monte-Carlo inputs from a counter-based generator (Philox4x32-10 keyed by `seed`, counter =
 * global rollout index), so results do not depend on how rollouts are sharded over GPUs.
 *   out[k][i] = lo[k] + (hi[k]-lo[k]) * U(seed, index_base+i, stream_id, k)      k < n_fields
 * out is [n_fields][B] fp32 SoA. */
int uavb_mc_uniform_f32(unsigned long long seed, long long index_base, int stream_id, int B, int n_fields,
                        const float* lo, const float* hi, float* out, void* stream);

/* BASELINE configs[1] mission generator (SURVEY 8(d) C2), fp64: first waypoint uniform in
 * [2,22]x[2,12]x[-5,-1]; each next = previous + step * u, u uniform on the sphere with z scaled by
 * 0.4, step ~ U(2,5) m; velocity ~ U(2,3) m/s.  waypoints_out [B][S+1][3], velocity_out [B]. */
int uavb_mc_missions_f64(unsigned long long seed, long long index_base, int B, int S,
                         double* waypoints_out, double* velocity_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * RRT* path planning for B missions, fp64, one warp per mission (SURVEY 8(f) rank 4).
 *
 * Replaces RRTStar(space_limits, start, goal, max_distance, max_iterations, obstacles).run() followed by
 * .best_path and .simplify_path(best_path) (uav_ac/planning/rrt.py:12-118): goal bias 0.15, neighbourhood radius
 * 1.5 x max_distance, coordinates rounded to 2 decimals, early stop after max_iterations/10 iterations without a better
 * path.  Random numbers come from Philox keyed by (seed, index_base + mission), so results do not depend on batching.
 *   space_limits [2][3] lower, upper (shared)      start, goal [B][3]      obstacles [n_obs][6] (shared) or NULL
 *   workspace    uavb_rrt_workspace_bytes(B, max_iterations) bytes of device memory
 *   path_out     [B][max_path][3] start -> goal,   path_len_out [B]
 *   simple_path_out / simple_len_out: greedy shortcut of the path (rrt.py:97-118); both NULL to skip
 *   cost_out [B] length of the path (inf when none), status_out [B]: 0 ok, 1 no path found (the reference raises),
 *   2 path longer than max_path;  stats_out [B][2] = iterations used, nodes in the best tree; may be NULL */
long long uavb_rrt_workspace_bytes(int B, int max_iterations);
int uavb_rrt_star_f64(const double* space_limits, const double* start, const double* goal, int B, double max_distance,
                      int max_iterations, const double* obstacles, int n_obs, unsigned long long seed, long long index_base,
                      void* workspace, double* path_out, int max_path, int* path_len_out, double* simple_path_out,
                      int* simple_len_out, double* cost_out, int* status_out, int* stats_out, void* stream);

/* RRTStar._segment_intersects_cuboid / _is_valid_connection (rrt.py:232-274) for n segments p[i] -> q[i]:
 * hit_out[i] = 1 when the segment intersects ANY of the n_obs boxes (exact slab test), else 0. */
int uavb_segments_hit_aabbs_f64(const double* p, const double* q, int n, const double* boxes, int n_obs, int* hit_out,
                                void* stream);

/* Measured FMA throughput of the device in TFLOP/s (2 flop per FMA), for the roofline denominators
 * that MEASURED_PEAKS.json does not carry.  Synchronous. */
int uavb_measure_fma_peak(int dev, double* fp32_tflops, double* fp64_tflops);

/* The same plus the fp32 rate of FMAs whose three sources are three DIFFERENT registers (x = y * z + x with nothing for the
 * operand reuse cache): a scheduler reads two register operands per cycle, so this is ~2/3 of fp32_tflops on sm_100 and the
 * practical ceiling of three-operand code such as the rollout's tick (profiles/r02_ffma2_probe.md).  Synchronous. */
int uavb_measure_fma_rates(int dev, double* fp32_tflops, double* fp32_three_operand_tflops, double* fp64_tflops);

/* ------------------------------------------------------------------------------------------------
 * Host-buffer (end-to-end) entry points: HOST pointers in and out, copies and synchronisation inside.
 */
int uavb_minsnap_solve_f64_host(const double* waypoints, const double* velocity, int B, int S,
                                double start_end_time_factor, double* coeffs_out, double* times_out,
                                int* status_out);

/* One mission flown by B drones, HOST buffers in and out -- the call a reference-side binding makes.
 * Replaces, for B drones at once, what uav_ac/main.py:main() and the headless loop of
 * tests/integration/test_mujoco_trajectory_tracking.py:11-36 do for one:
 *     trajectory = _generate_mission_trajectory(waypoints, obstacles, velocity, quad.dt * frequency)   (main.py:73-84)
 *     for target in trajectory: for _ in range(frequency): trajectory_controller.step(); simulation.step()
 *     final distance to goal / collision flag / tracking error                                          (main.py:115-120)
 * The mission is planned on the device (both tables through the obstacle-correction loop uavb_minsnap_correct_f64, then the
 * table geometry), every drone flies it in the
 * persistent rollout kernel (K2) with its own Monte-Carlo overrides, and the per-rollout metrics
 * (and optionally the final states) are copied back.  Synchronous. */
typedef struct uavb_mission_host {
  int B;                        /* drones                                                                */
  int n_waypoints;              /* rows of `waypoints`                                                   */
  int n_takeoff_waypoints;      /* leading waypoints of the first (take-off) table: 2 for main.py:80-81;
                                   the second table starts at waypoint n_takeoff_waypoints-1 (:82-83).
                                   0 = a single table over all waypoints                                  */
  const double* waypoints;      /* [n_waypoints][3] NED                                                  */
  double velocity;              /* config.ini [SIM_FLIGHT] velocity                                      */
  double start_end_time_factor; /* MinimumSnap.START_END_TIME_FACTOR (1.5)                               */
  int frequency;                /* config.ini [DEFAULT] frequency: inner ticks per outer period          */
  int n_ticks;                  /* ticks to fly; 0 = the whole table (frequency * rows)                  */
  int thrust_frame_lag;         /* 1 = headless loop, 0 = viewer path (SURVEY 3.2)                       */
  uavb_vehicle veh;
  const float* mc_mass;         /* [B]      optional per-drone overrides, SoA, NULL = veh defaults        */
  const float* mc_inertia;      /* [3][B]                                                                */
  const float* mc_gains;        /* [UAVB_N_GAINS][B]                                                     */
  const float* mc_wind;         /* [3][B]   N, world frame (extension)                                   */
  const float* aabbs;           /* [n_obs][6] or NULL                                                    */
  int n_obs;
  const double* start;          /* [3] or NULL = waypoints[0]                                            */
  const double* goal;           /* [3] or NULL = last waypoint                                           */
  const double* plan_aabbs;     /* [n_obs][6] fp64 boxes for the planner's correction loop (the reference tests its
                                   fp64 obstacle array, minimum_snap.py:84-87); NULL = `aabbs` widened to double */
  int no_correction;            /* 0 = plan like MinimumSnap.get_trajectory() with obstacles (midpoint insertion,
                                   minimum_snap.py:63-95); 1 = fly the waypoints as given                         */
} uavb_mission_host;
int uavb_fly_mission_host(const uavb_mission_host* mission, float* metrics_out /* [B][UAVB_N_METRICS] */,
                          float* state_out /* [13][B] or NULL */, int* n_ticks_out /* or NULL */);

#ifdef __cplusplus
}
#endif
#endif /* UAVB_H */
