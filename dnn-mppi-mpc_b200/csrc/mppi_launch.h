// Launch entry points of mppi_kernels.cu used by the C-ABI host code (mppi_api.cu).
#pragma once
#include <cuda_runtime.h>
struct TickArgs;
struct SceneRec;
// stash: 0 regenerate, 1 noise stash, 2 stash + time-parallel rollout; scene: the per-robot-scene instantiation (a.scene /
// a.scene_mask; Philox noise, stash 0 or 1, the combinations mppi_set_robot_* accept -- cudaErrorInvalidValue otherwise)
cudaError_t mppi_launch_tick(const TickArgs &a, int model, int coll, int cost_kind, bool sum, bool inj, int stash, dim3 grid,
                             cudaStream_t st, bool scene = false);
size_t mppi_tick_dyn_smem(int T, int stash);
cudaError_t mppi_launch_strict(const TickArgs &a, int model, int coll, bool sum, bool inj, const unsigned *bp_n,
                               const int *bp_s, int nbp, int k_first, unsigned check_from,
                               unsigned long long *first_change, cudaStream_t st);
cudaError_t mppi_launch_merge(const TickArgs &a, const float *triples, int G, cudaStream_t st);
cudaError_t mppi_launch_p2p_barrier(const TickArgs &a, unsigned long long count, cudaStream_t st);
cudaError_t mppi_launch_traj(const TickArgs &a, int model, const float *rec, float *d_opt, float *d_samp,
                             const int *d_sel, int n_sel, int shift, cudaStream_t st);
// mppi_spline.cu: per-robot courses from waypoints (calc_spline_course on the device)
#define MPPI_SPLINE_MAX_WAYPOINTS 32
cudaError_t mppi_launch_spline(const float *d_wx, const float *d_wy, int n_robots, int n_wp, double ds, int max_pts,
                               float4 *d_paths, int *d_path_len, cudaStream_t st);
// mppi_topn.cu: ascending (cost, sample index) order of K costs -- np.argsort(S) of the viewers
size_t mppi_sort_costs_temp_bytes(int K);
cudaError_t mppi_sort_costs(const float *d_S, int K, float *d_S_sorted, int *d_idx_sorted, int *d_iota, void *d_temp,
                            size_t temp_bytes, cudaStream_t st);
cudaError_t mppi_launch_noise(const TickArgs &a, float *d_out, int robot, cudaStream_t st);
int mppi_tick_occupancy(int model, int coll, int cost_kind, bool sum, bool inj, int window, int T, int stash, bool scene = false);
// Installs per-robot scene components into d_scene[R] (in stream order; FP64 conversions of refresh_obstacle_args).
//   obstacles: d_obs (R, m, ncol) float32, ncol 3 [x, y, r] (circle: r2 = (rr_base + r)^2 with rr_base = robot radius * margin;
//   footprint: r2 = r^2; far2 = ((diag + r) * 1.001 + 1e-3)^2) or 4 [x, y, vx, vy]; d_count (R) int32 or null
cudaError_t mppi_launch_scene_obstacles(const float *d_obs, const int *d_count, int R, int m, int ncol, bool circle,
                                        double rr_base, double diag, SceneRec *d_scene, cudaStream_t st);
cudaError_t mppi_launch_scene_goals(const float *d_goal, int R, int n, SceneRec *d_scene, cudaStream_t st);
