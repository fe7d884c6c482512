/* libmppi_b200.so -- C ABI of the B200-native MPPI engine.
 *
 * The reference (SokhengDin/DNN-MPPI-MPC) has no FFI layer: its boundary is the Python
 * class surface of controllers/mppi_*.py.  Each entry point below names the reference
 * code it replaces (file:line relative to the reference tree); the Python shim in
 * dnn-mppi-mpc_b200/mppi_b200/ binds these with ctypes and re-exposes the reference's
 * class/method names (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; no C++/torch types cross this boundary.
 *   - pointers named d_* are DEVICE pointers (e.g. torch.Tensor.data_ptr()); all others
 *     are HOST pointers.  The caller owns every pointer it passes in; the library owns
 *     the handle's device scratch for the handle's lifetime.
 *   - every call returns an int status (0 = MPPI_OK, <0 = MPPI_E_*); nothing throws or
 *     aborts across the ABI.  mppi_last_error(h) returns the last CUDA/NCCL message.
 *   - a handle is bound to one device and one stream and is not thread-safe; distinct
 *     handles are independent.
 *   - there is NO CPU fallback: without a CUDA device mppi_create fails with MPPI_E_CUDA.
 */
#ifndef MPPI_B200_H
#define MPPI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPPI_ABI_VERSION 3

typedef struct mppi_handle_s *mppi_handle_t;

enum mppi_status {
    MPPI_OK = 0,
    MPPI_E_BADARG = -1,       /* invalid configuration / null pointer / size out of range */
    MPPI_E_CUDA = -2,         /* CUDA runtime error (message via mppi_last_error) */
    MPPI_E_NCCL = -3,         /* NCCL error */
    MPPI_E_STATE = -4,        /* call order: path / nominal / MLP weights not set yet */
    MPPI_E_UNSUPPORTED = -5,  /* mode combination not implemented by this build */
    MPPI_E_NOMEM = -6,
    MPPI_E_NUMERIC = -7       /* non-finite sample costs (NaN/inf state or residual, missed cluster hand-off): tick NOT applied */
};

enum mppi_model {
    MPPI_MODEL_DIFFDRIVE = 0,      /* controllers/mppi_differential_drive.py:182-198 */
    MPPI_MODEL_BICYCLE = 1,        /* controllers/mppi_race_car_obstacle.py:200-214, u = [steer, accel] */
    MPPI_MODEL_DIFFDRIVE_MLP = 2   /* unicycle + dnn/simple_mlp.py residual (SURVEY.md 3.4) */
};
enum mppi_cost_mode { MPPI_COST_LAST = 0 /* :124 assigns (Q1) */, MPPI_COST_SUM = 1 /* race-car :94 */ };
enum mppi_waypoint_mode { MPPI_WP_STRICT = 0 /* :228,:244 mutate the index (Q3) */, MPPI_WP_FROZEN = 1 };
enum mppi_filter_kind { MPPI_FILTER_DIFFDRIVE = 0 /* :257-271 */, MPPI_FILTER_RACECAR = 1 /* race-car :228-239 */ };
/* What a state is scored against (A9).  PATH: nearest waypoint of `ref_path` (controllers/mppi_*.py).
 * GOAL: squared distance to `goal` plus squared wrapped bearing error, the goal-point diff-drive MPPI of
 * test/mppi_differential_drive_obs.py:202-232 (no waypoint search, no carried index).
 * TARGET_SOFT: quadratic error to a target pose + control effort + exponential soft penalty around MOVING circular
 * obstacles, the running cost of test/test_mppi_diff_obs.py:14-20,44-66 (summed over the horizon). */
enum mppi_cost_kind { MPPI_COSTKIND_PATH = 0, MPPI_COSTKIND_GOAL = 1, MPPI_COSTKIND_TARGET_SOFT = 2 };
enum mppi_collision {
    MPPI_COLLISION_NONE = 0,
    MPPI_COLLISION_CIRCLE = 1,     /* controllers/mppi_differential_drive_obs.py:301-313 */
    MPPI_COLLISION_FOOTPRINT = 2   /* controllers/mppi_race_car_obstacle.py:255-274 */
};

#define MPPI_MAX_T 128
#define MPPI_MAX_WINDOW 256
#define MPPI_MAX_OBSTACLES 16

/* Mirrors every constructor kwarg of the reference controllers plus the constants they
 * hard-code (controllers/mppi_differential_drive.py:44-85,204; mppi_race_car_obstacle.py:11-62,175). */
typedef struct {
    int32_t abi_version;      /* = MPPI_ABI_VERSION */
    int32_t device;           /* CUDA device ordinal */
    int32_t model;            /* enum mppi_model */
    int32_t K;                /* num_samples_K / number_of_samples_K: samples THIS handle rolls out */
    int32_t T;                /* num_horizons_T / horizon_step_T, <= MPPI_MAX_T */
    int32_t n_robots;         /* 1, or R independent controllers solved in one launch */
    int32_t window;           /* SEARCH_IDX_LEN: 20 / 200, <= MPPI_MAX_WINDOW */
    int32_t cost_mode;        /* enum mppi_cost_mode */
    int32_t waypoint_mode;    /* enum mppi_waypoint_mode */
    int32_t filter_kind;      /* enum mppi_filter_kind */
    int32_t yaw_wrap;         /* 1: yaw = (yaw + 2pi) mod 2pi inside the cost (race-car :151) */
    int32_t collision;        /* enum mppi_collision */
    int32_t K_global;         /* total samples over all ranks (== K when not sharded) */
    int32_t k_offset;         /* global index of this handle's first sample */
    int32_t clamp_nominal;    /* 1: clamp the updated nominal in place before the shift -- the side effect of the
                                 visualisation replay (quirk Q9: mppi_differential_drive.py:145-148, race-car :112-115) */
    int32_t cost_kind;        /* enum mppi_cost_kind */
    double dt;                /* delta_t */
    double wheel_base;
    double u_max[2];          /* (max_speed, max_omega) or (max_steer_abs, max_accel_abs) */
    double param_exploration; /* explore/exploit split (Q6) */
    double param_lambda;
    double param_alpha;       /* gamma = lambda * (1 - alpha) */
    double temperature;       /* softmax temperature: param_exploration (diff-drive, Q2) or param_lambda */
    double sigma[4];          /* row-major 2x2 noise covariance */
    double stage_w[4];
    double term_w[4];
    double margin;            /* safety_margin_rate / collision_safety_margin_rat */
    double robot_radius;      /* 0.5 (mppi_differential_drive_obs.py:303) */
    double vehicle_l;         /* 4.0 (mppi_race_car_obstacle.py:54) */
    double vehicle_w;         /* 3.0 (mppi_race_car_obstacle.py:53) */
    double goal[4];           /* GOAL: goal_point (x, y) (test/mppi_differential_drive_obs.py:65);
                                 TARGET_SOFT: desired pose (x, y, yaw) (test/test_mppi_diff_obs.py:45) */
    double ctrl_w[2];         /* TARGET_SOFT: diagonal of R (test/test_mppi_diff_obs.py:48) */
    double soft_obs_weight;   /* TARGET_SOFT: obstacle_weight 100.0 (:57) */
    double soft_obs_safety;   /* TARGET_SOFT: safety_distance 2.0 (:56) */
} mppi_config_t;

typedef struct {
    float last_step_ms;       /* device time of the last mppi_step (CUDA events), timing enabled only */
    float last_rollout_ms;
    float last_update_ms;
    int32_t last_passes;      /* strict mode: rollout passes of the last tick */
    int32_t launches;         /* kernels launched by this handle since creation */
} mppi_timings_t;

typedef struct {
    float rho;                /* min cost of the tick */
    float eta;                /* sum of unnormalised weights */
    float ess;                /* effective sample size (sum w)^2 / sum w^2 */
    int32_t min_collisions;   /* fewest collided evaluations among the samples */
    int32_t idx;              /* carried waypoint index after the tick */
    float u_first[2];         /* row 0 of the updated nominal BEFORE the shift: what a textbook MPPI (pytorch_mppi's
                                 `command`, test/test_mppi_diff_obs.py:80) applies; the reference classes return the
                                 post-shift row 0 instead (quirk Q8), which is what mppi_step hands back */
} mppi_stats_t;

/* lifecycle -- replaces MPPIAlgorithms.__init__ (controllers/mppi_differential_drive.py:44-85)
 * and MPPIRacecarController.__init__ (controllers/mppi_race_car_obstacle.py:11-62) */
int mppi_create(const mppi_config_t *cfg, mppi_handle_t *out);
int mppi_destroy(mppi_handle_t h);
void mppi_default_config(mppi_config_t *cfg);
const char *mppi_strerror(int status);
const char *mppi_last_error(mppi_handle_t h);
int mppi_set_stream(mppi_handle_t h, void *cuda_stream);
int mppi_synchronize(mppi_handle_t h);

/* `self.ref_path` (N,3) [x,y,yaw] or (N,4) [x,y,yaw,v], row-major doubles
 * (mppi_differential_drive.py:64; re-assigned after construction at mppi_race_car_obstacle.py:332) */
int mppi_set_ref_path(mppi_handle_t h, const double *path, int32_t n, int32_t ncol);
/* Fleets with ONE PATH PER ROBOT (batched handles, SURVEY.md 8f row 4): robot r's course is generated on the device
 * from its n_wp waypoints by the reference's own course generator -- `calc_spline_course(x, y, ds)`
 * (path_generator/cubic_spline_planner.py:311-323: arclength-parameterised natural cubic spline, sampled every ds,
 * yaw = atan2 of the first derivatives; FP64 like the reference) -- and installed as that robot's `ref_path`.
 *   d_wx, d_wy   device (n_robots, n_wp) float32 waypoint coordinates, 2 <= n_wp <= 32
 *   max_points   capacity per robot; MPPI_E_BADARG if a course needs more than that
 * mppi_set_ref_path afterwards returns the handle to one shared path.  Frozen waypoint mode, diff-drive models. */
int mppi_set_ref_paths_spline(mppi_handle_t h, const float *d_wx, const float *d_wy, int32_t n_wp, double ds,
                              int32_t max_points);
/* The path robot `robot` follows, as (n, 4) float32 rows [x, y, yaw, v]: n to *n_out, min(n, capacity) rows to
 * path_out (host, may be NULL to query n). */
int mppi_get_ref_path(mppi_handle_t h, int32_t robot, float *path_out, int32_t capacity, int32_t *n_out);
/* `self.obstacle_circles` (M,3) [x,y,r] (mppi_race_car_obstacle.py:57) */
int mppi_set_obstacles(mppi_handle_t h, const double *xyr, int32_t m);
/* `self.goal_point` (x, y) of the goal-point controller (test/mppi_differential_drive_obs.py:65), or the desired
 * pose (x, y, yaw) of the TARGET_SOFT cost (test/test_mppi_diff_obs.py:45); n = 2 or 3 doubles */
int mppi_set_goal(mppi_handle_t h, const double *goal, int32_t n);
/* TARGET_SOFT: circular soft obstacles moving at constant velocity, position at horizon step t (time t*dt) =
 * pos + vel * (t*dt)  (`get_obstacle_positions`, test/test_mppi_diff_obs.py:14-20).  pos_xy, vel_xy: (M,2) doubles */
int mppi_set_moving_obstacles(mppi_handle_t h, const double *pos_xy, const double *vel_xy, int32_t m);
/* Fleets with their OWN SCENE PER ROBOT (batched handles).  Each call enqueues one small kernel on the handle's stream that
 * converts the caller's rows into a handle-owned per-robot table (r2 / far2 in FP64, as mppi_set_obstacles computes them);
 * the caller may overwrite its buffers with work ordered after the call on that stream, and no host synchronisation takes
 * place.  Goals and obstacles are independent components: the matching shared setter (mppi_set_goal, mppi_set_obstacles,
 * mppi_set_moving_obstacles) returns that component to the shared value.  mppi_step_batched and mppi_run_closed_loop run
 * the per-robot scene (the closed-loop graph holds the table's address only, so a re-install between calls takes effect
 * without re-instantiating it); while a component is installed every other tick entry point (mppi_step, mppi_step_async,
 * mppi_rollout_costs, mppi_reduce_update, the trajectory viewers, mppi_comm_*) returns MPPI_E_STATE.
 * MPPI_E_STATE: a component the handle's kind does not have; MPPI_E_UNSUPPORTED: strict waypoint mode, learned dynamics,
 * sample sharding, or a model / collision / cost kind without a per-robot-scene kernel (built: diff-drive + circles and
 * bicycle + footprint on a path, GOAL without obstacles or with circles, TARGET_SOFT).
 *   d_obs    device (n_robots, m, ncol) float32, 0 <= m <= MPPI_MAX_OBSTACLES;
 *            ncol = 3: static circles [x, y, r] (CIRCLE / FOOTPRINT collision, like mppi_set_obstacles);
 *            ncol = 4: moving soft obstacles [x, y, vx, vy] (TARGET_SOFT, like mppi_set_moving_obstacles)
 *   d_count  device n_robots int32 (robot r uses its first d_count[r] rows, clamped into [0, m]) or NULL (all m) */
int mppi_set_robot_obstacles(mppi_handle_t h, const float *d_obs, const int32_t *d_count, int32_t m, int32_t ncol);
/* One goal PER ROBOT: d_goal device (n_robots, n) float32, n = 2 (GOAL: goal_point) or 3 (TARGET_SOFT: target pose). */
int mppi_set_robot_goals(mppi_handle_t h, const float *d_goal, int32_t n);
/* `self.u_prev` (T,2) per robot (mppi_differential_drive.py:82) -- host float arrays of n_robots*T*2 */
int mppi_set_nominal(mppi_handle_t h, const float *u);
int mppi_get_nominal(mppi_handle_t h, float *u);
/* `self.prev_way_point_idx` / `prev_waypoints_idx` (mppi_differential_drive.py:85) -- n_robots ints */
int mppi_set_waypoint_idx(mppi_handle_t h, const int32_t *idx);
int mppi_get_waypoint_idx(mppi_handle_t h, int32_t *idx);
/* weights of dnn/simple_mlp.py (3-512-512-512-3), row-major float32 [out][in] like nn.Linear */
int mppi_set_mlp(mppi_handle_t h, const float *const W[4], const float *const b[4]);
/* The reference's TRAINED residuals (saved_models/mlp_diff*.pth; class at simulation/bullet_differential_drive_dnn.py:37-60,
 * training at train/train_diff_mlp.py:13-36,72-103): n_in = 5 inputs [x, y, yaw, v, w] -> 512 -> n_hidden x tanh(512) -> 3,
 * added to the unicycle right-hand side like controllers/mpc_mlp_differential_drive.py:65-71, with the StandardScaler
 * pre/post-processing of test/test_diff_dyna_eval.py:54-56:
 *     x+ = x + dt * ( f(x, u) + out_scale * MLP(([x; u] - in_mean) / in_scale) + out_mean ).
 * W / b: n_hidden + 2 nn.Linear tensors [out][in] (input layer n_in -> 512 first, output layer 512 -> 3 last);
 * in_mean / in_scale: n_in doubles (state scaler then control scaler) or NULL; out_mean / out_scale: 3 doubles or NULL.
 * n_in = 3 is dnn/simple_mlp.py (mppi_set_mlp).  n_hidden = 2 (simulation/bullet_differential_drive_dnn.py:43-45,
 * mlp_diff.pth, mlp_diff_300x100.pth, mlp_diff_300x100_v2.pth) or 3 (train/train_diff_mlp.py:19-21,
 * mlp_diff_300x100_3l.pth, mlp_diff_300x100_3l_mppi.pth: a second tensor-core GEMM per step); MPPI_E_UNSUPPORTED
 * otherwise. */
int mppi_set_mlp_ex(mppi_handle_t h, int32_t n_in, int32_t n_hidden, const float *const *W, const float *const *b,
                    const double *in_mean, const double *in_scale, const double *out_mean, const double *out_scale);

/* One control tick -- replaces the body of `_calc_input_control` (mppi_differential_drive.py:87-165)
 * / `_calc_control_input` (mppi_race_car_obstacle.py:65-131): index update, noise, K x T rollout,
 * costs, weights, weighted noise, filter, nominal update and shift.
 *   x0        host, nx doubles (observed state)
 *   d_eps     device (K,T,2) float32 injected noise, or NULL -> Philox4x32-10 with (seed, tick)
 *   u0_out    host, 2 floats: the returned control (post-shift row 0, quirk Q8); may be NULL
 *   useq_out  host, T*2 floats: the returned (shifted) sequence; may be NULL */
int mppi_step(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick,
              float *u0_out, float *useq_out);
/* Same tick without any host copy: results stay on the device (nominal, stats). */
int mppi_step_async(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick);
/* K1 alone: index update + rollout + costs -> d_S (K float32, device).  Does not touch the nominal.
 * Replaces the loop at mppi_differential_drive.py:111-126 / mppi_race_car_obstacle.py:82-96. */
int mppi_rollout_costs(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed,
                       uint64_t tick, float *d_S);
/* K2 alone: weights + weighted noise + filter + update + shift from given costs
 * (mppi_differential_drive.py:129-141,162-163,167-180,257-271).  w_eps_out: host T*2 raw weighted noise. */
int mppi_reduce_update(mppi_handle_t h, const float *d_S, const float *d_eps, uint64_t seed,
                       uint64_t tick, float *u0_out, float *useq_out, float *w_eps_out);
/* The exact noise tensor (K,T,2) the Philox path consumes for (seed, tick) -- replaces
 * `_calc_epsilon` (mppi_differential_drive.py:273-283) and lets the oracle be fed the same noise. */
int mppi_generate_noise(mppi_handle_t h, uint64_t seed, uint64_t tick, float *d_eps_out);
/* Same for robot `robot` of a batched handle (its Philox stream is keyed by the robot index). */
int mppi_generate_noise_robot(mppi_handle_t h, uint64_t seed, uint64_t tick, int32_t robot, float *d_eps_out);
int mppi_get_stats(mppi_handle_t h, mppi_stats_t *out);   /* robot 0 */
/* Visualisation outputs of the LAST tick (A16: mppi_differential_drive.py:144-159, mppi_race_car_obstacle.py:111-125):
 * the replay of the updated (pre-shift) nominal and of every sample's clamped controls, both with the reference's
 * `t-1` indexing.  Call right after mppi_step with the same x0 / d_eps / seed / tick.
 * Learned dynamics (MPPI_MODEL_DIFFDRIVE_MLP): the same controls are replayed through the tick's own tensor-core MLP
 * rollout, so a replayed state is the state the tick scored (fp16 hidden layers, hardware tanh; DESIGN.md 3.4).  The
 * nominal, the waypoint index and the tick's fault word are not touched; a missed cluster hand-off of the replay
 * returns MPPI_E_NUMERIC.  Fleets (n_robots > 1) return MPPI_E_UNSUPPORTED.
 *   optimal_out  host, T*nx floats, or NULL;   d_sampled_out  device, K*T*nx floats, or NULL */
int mppi_get_trajectories(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick,
                          float *optimal_out, float *d_sampled_out);

/* Top-N viewer (SURVEY.md 8f row 2): the n_top lowest-cost samples of the LAST tick in ascending cost order
 * (`sorted_idx = np.argsort(S)`, controllers/mppi_differential_drive.py:153; `torch.argsort(self.cost_total)
 * [:num_top_samples]` with num_top_samples = max(10, K/10), test/test_mppi_diff_obs.py:102-104) replayed from x0,
 * instead of all K trajectories (600 MB at K = 1M, H = 50).  mppi_set_keep_costs(h, 1) makes every following tick
 * keep its per-sample costs (4 bytes per sample); call mppi_get_top_trajectories right after mppi_step with the same
 * x0 / d_eps / seed / tick.  Learned dynamics: as mppi_get_trajectories (the n_top rows and the nominal are replayed
 * through the tick's MLP rollout); the tick keeps its costs in the same buffer the sort reads.
 *   index_shift   1: controls indexed t-1, last row first, like the reference classes (A16);
 *                 0: controls indexed t (test/test_mppi_diff_obs.py:94,108)
 *   optimal_out   host T*nx floats, replay of the updated pre-shift nominal, or NULL
 *   d_traj_out    device (n_top, T, nx) float32;  d_idx_out device n_top int32 sample indices or NULL;
 *   d_cost_out    device n_top float32 costs (smooth + 1e10 * collided evaluations) or NULL */
int mppi_set_keep_costs(mppi_handle_t h, int32_t enabled);
int mppi_get_top_trajectories(mppi_handle_t h, const double *x0, const float *d_eps, uint64_t seed, uint64_t tick,
                              int32_t n_top, int32_t index_shift, float *optimal_out, float *d_traj_out,
                              int32_t *d_idx_out, float *d_cost_out);

/* On-device closed loop (A17): n_ticks control ticks with the plant step applied on the device between them, no
 * host round trip per tick; the n ticks run as ONE CUDA graph (instantiated on first use, re-launched afterwards).
 * plant 0 = DifferentialDrive.update_state (controllers/mppi_differential_drive.py:33-40, Euler unicycle, unclamped u0);
 * plant 1 = Vehicle.update (models/vehicle.py:95-110, clamp then Euler bicycle).  Tick i uses the Philox stream
 * (seed, tick0 + i).  Frozen waypoint mode.  FLEETS: a handle created with n_robots = R runs R independent closed loops
 * (own state, nominal, waypoint index and Philox stream per robot; R copies of the loop at :305-367) in the same launches.
 *   x0           host, R*nx doubles
 *   states_out   host, (n_ticks+1)*R*nx floats: [tick][robot][nx], row 0 = x0
 *   controls_out host, n_ticks*R*2 floats: [tick][robot][2] (may be NULL) */
int mppi_run_closed_loop(mppi_handle_t h, const double *x0, int32_t n_ticks, uint64_t seed, uint64_t tick0,
                         int32_t plant, float *states_out, float *controls_out);

/* Batched multi-robot tick: n_robots independent controllers in one launch (no reference
 * equivalent; R copies of the loop at mppi_differential_drive.py:111-141).
 *   d_x0  device (R, nx) float32;  d_u0_out device (R, 2) float32 (may be NULL)
 * A robot whose sample costs are not finite (NaN state) is not updated: its u0 row reads NaN, its nominal and waypoint
 * index stay as they were, the other robots are unaffected, and the next mppi_synchronize returns MPPI_E_NUMERIC naming
 * the first such robot (mppi_run_closed_loop likewise, with that robot's log rows NaN from the faulted tick on). */
int mppi_step_batched(mppi_handle_t h, const float *d_x0, uint64_t seed, uint64_t tick, float *d_u0_out);

/* Sample sharding across GPUs: each rank owns K of K_global samples; one exchange of
 * (min cost, sum w, sum w*eps) per tick.  `nccl_unique_id` is the 128-byte ncclUniqueId. */
int mppi_comm_get_unique_id(void *out128);
int mppi_comm_init(mppi_handle_t h, const void *nccl_unique_id, int32_t rank, int32_t world);
/* The same exchange fused INTO the tick kernel over NVLink peer memory (no NCCL call, one launch per tick): every
 * rank's last CTA writes each word of its (min, sum w, sum w*eps) triple straight into every peer's exchange buffer as
 * one 8-byte store (tick sequence number, float bits) -- the flag travels with the datum, so there is no system fence
 * and no second round trip -- polls its own buffer until every rank's words carry this tick's number, and merges them
 * in rank order (bit-identical nominal on all ranks).  Set-up: each rank exports its buffer with mppi_comm_p2p_export
 * (64-byte cudaIpcMemHandle_t), the handles are all-gathered by the caller (any transport) and handed to
 * mppi_comm_p2p_open as world*64 bytes in rank order.  One process per GPU, all GPUs on one NVLink domain.
 * A peer that has not published within MPPI_P2P_TIMEOUT_MS (environment, default 2000) fails THAT tick: the nominal
 * and the waypoint index are left untouched and mppi_step / mppi_synchronize return MPPI_E_NCCL once. */
#define MPPI_MAX_PEERS 8
int mppi_comm_p2p_export(mppi_handle_t h, int32_t world, void *ipc_handle_out64);
int mppi_comm_p2p_open(mppi_handle_t h, const void *ipc_handles, int32_t rank, int32_t world);
/* Device-side barrier of the ranks of a fused exchange, enqueued on the handle's stream (asynchronous; no host round trip, no
 * NCCL call): the GPUs leave it within a microsecond of each other.  bench.py aligns the ranks with it in front of each
 * timed tick so the L2 flush of a slower GPU is not billed to the others' tick. */
int mppi_comm_p2p_barrier(mppi_handle_t h);
/* Diagnostics of the last fused exchange on this rank: %globaltimer stamps (ns) of [0] local merge done, [1] words
 * stored, [2] every rank's words seen, [3] nominal updated.  [2]-[1] is the wait for the slowest rank. */
int mppi_comm_p2p_trace(mppi_handle_t h, uint64_t stamps_out[4]);

/* Diagnostics, no reference counterpart: per-CTA %globaltimer stamps (ns) of the LAST single-robot tick -- out[2b] CTA b
 * entered the kernel, out[2b+1] its rollouts ended; after the n CTAs: out[2n] partials merged, out[2n+1] nominal updated
 * (last CTA).  Shows where a tick's time outside the rollouts goes (profiles/).  *n_ctas_out is the grid width (CTAs per
 * robot) of the last traced launch, which depends on the rollout path that tick took (regenerate, stash, time-parallel). */
int mppi_set_trace(mppi_handle_t h, int32_t enabled);
int mppi_get_trace(mppi_handle_t h, uint64_t *out, int32_t capacity, int32_t *n_ctas_out);

/* Every device buffer of a handle carries a 256-byte guard zone; returns how many were overwritten (0 = no kernel wrote
 * past a buffer), < 0 on error.  Bounds evidence for pools where compute-sanitizer cannot run (profiles/). */
int mppi_debug_check_guards(mppi_handle_t h);
int mppi_set_timing(mppi_handle_t h, int32_t enabled);
int mppi_get_timings(mppi_handle_t h, mppi_timings_t *out);
int mppi_abi_version(void);
/* Measurement aid, no reference counterpart: achieved FP32 FMA throughput (TFLOP/s, best of 3) of a register-only FFMA
 * (packed = 0) or FFMA2 (packed = 1) loop filling every SM of `device` -- the measured denominator of the FP32 roofline the
 * analytic-dynamics kernels are bound by (SURVEY.md 8d; MEASURED_PEAKS.json has no FP32 entry). */
int mppi_probe_fp32_peak(int32_t device, int32_t packed, double *tflops_out);
/* Measurement aid: out[i] = the hardware tanh (tanh.approx.f32, MUFU.TANH) of in[i], n HOST floats each -- the activation
 * the learned-dynamics kernel applies where dnn/simple_mlp.py:20-21 calls torch.tanh; lets the parity tests state its
 * distance from the exact function instead of assuming it. */
int mppi_probe_tanh(int32_t device, const float *in, float *out, int32_t n);
/* Host-side view of the learned-dynamics kernel's balanced schedule (no reference counterpart, no GPU needed): the first
 * unit-step, in unit-major order u * T + t, that cluster `c` of `n_clusters` owns when `n_units` units (quads of 4 tiles in the
 * ping-pong schedule, pairs of 2 tiles otherwise) x T timesteps are dealt evenly; c = n_clusters gives the total.  The same
 * function the kernel evaluates, exported so the partition can be checked without a device.  Returns -1 on bad arguments. */
int mppi_mlp_schedule_cut(int32_t c, int32_t n_clusters, int32_t n_units, int32_t T);

#ifdef __cplusplus
}
#endif
#endif /* MPPI_B200_H */
