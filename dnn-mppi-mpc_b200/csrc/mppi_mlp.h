// Learned-dynamics rollout (K3): unicycle + simple_mlp residual, tcgen05 tensor-core MLP.
#pragma once
#include <cuda_runtime.h>
struct TickArgs;
// Balanced K3 schedule: first unit-step (unit-major index u * T + t) of cluster c when n_units units x T timesteps are dealt
// over n_clusters clusters; cuts fall on even timesteps (a Philox call yields the noise of two).  Shared by the kernel and
// the host-side check (mppi_mlp_schedule_cut).
#ifdef __CUDACC__
__host__ __device__
#endif
inline int mlp_bal_cut(int c, int n_clusters, int n_units, int T) {
    if (c >= n_clusters) return n_units * T;
    const long long raw = (long long)c * n_units * T / n_clusters;
    const int g = (int)(raw / T), t = (int)(raw % T) & ~1;
    return g * T + t;
}
struct MlpState;
MlpState *mlp_create(int K, int T);
void mlp_destroy(MlpState *m);
// n_in = 3 (state) or 5 (state + control); n_hidden = 2 or 3 tanh layers (W / b: n_hidden + 2 layers); scaler pointers
// may be null (identity)
cudaError_t mlp_set_weights(MlpState *m, int n_in, int n_hidden, const float *const *W, const float *const *b, const double *in_mean,
                            const double *in_scale, const double *out_mean, const double *out_scale, cudaStream_t st);
// index update + K x T rollout through the MLP + costs -> d_S; returns 0 on success
int mlp_rollout_costs(MlpState *m, const TickArgs &a, bool sum, const float *d_eps, float *d_S, cudaStream_t st);
// Replay (trajectory viewers): a.K rows, row k applies the controls d_ctl (K, T, 2) -- already clamped, so the rollout's own
// clamp leaves them exact -- through the same learned step as the tick.  d_out receives K costs (scratch: they are scored against
// whatever nominal `a` holds) followed by the state after every step, (K, T, 3).  A missed cluster hand-off raises *d_fault
// instead of the handle's fault word.  Returns 0 on success
int mlp_rollout_states(MlpState *m, const TickArgs &a, const float *d_ctl, float *d_out, unsigned int *d_fault, cudaStream_t st);
// true (and cleared) if a cluster hand-off of the balanced schedule was missed since the last call
bool mlp_take_fault(MlpState *m, cudaStream_t st);
// number of hand-off buffers whose guard zone was overwritten (0 = clean)
int mlp_check_guards(MlpState *m);
