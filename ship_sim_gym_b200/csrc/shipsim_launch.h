// shipsim_launch.h -- host-visible launch wrappers implemented in shipsim_kernels.cu
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace shipsim {

struct StepParams;
struct EdgeD;
constexpr int kThreads = 128;

struct LaunchShape { int lanes_per_env, threads, blocks, window; };

cudaError_t launch_step(const StepParams &p, int lanes_per_env, cudaStream_t stream, LaunchShape *shape);
// time-parallel variant (shipsim_window.cu): `window` = 4, 8, 16 or 32 speculated steps per env; `chain`: a chained
// launch (log-free, p.chain_* bound), which may overlap the previous kernel of the stream
cudaError_t launch_window(const StepParams &p, int window, cudaStream_t stream, LaunchShape *shape, bool chain);
cudaError_t launch_reset(const StepParams &p, const uint8_t *mask, const int *scenario, int first, float4 *obs,
                         cudaStream_t stream);
cudaError_t launch_build_grid(const double *hull_xy, const int *hull_n, int n_scen, int maxv_in, double gx0, double gy0,
                              double cw, double ch, double reach, double touch_margin, uint4 *grid, cudaStream_t stream);
cudaError_t launch_build_spawn_rows(const StepParams &p, float4 *rows, cudaStream_t stream);
cudaError_t launch_gen_scenarios(unsigned long long seed, int n_scen, double W, double H, int map_N, double width_frac, double *hull_xy,
                                 int *hull_n, double *goals, cudaStream_t stream);
cudaError_t launch_pack_bank(double *hull_xy, const int *hull_n, const double *goals, int n_scen, int maxv, int stride4, float4 *bank,
                             EdgeD *edges, cudaStream_t stream);
cudaError_t launch_max_hull(const int *hull_n, int n, int *out, cudaStream_t stream);
cudaError_t launch_clamp_scenarios(float4 *state, int N, int n_scen, cudaStream_t stream);
cudaError_t launch_compact_frames(const float4 *frames, const float4 *prev0, const float *rew, const uint8_t *done, int N, int env0, int kc,
                                  float step_penalty, uint4 *rec, unsigned *off, float *var, unsigned var_cap, unsigned *counter,
                                  cudaStream_t stream);
cudaError_t launch_history_rows(const float4 *frames, const float4 *prev0, const uint8_t *done, int N, int nd, int kc, int cut, float4 *rows,
                                cudaStream_t stream);
cudaError_t launch_frame(const StepParams &p, float4 *out, cudaStream_t stream);
cudaError_t launch_gae(const float *rew, const float *val, const unsigned char *done, int T, int N, float gamma, float lam, float *adv, float *ret,
                       cudaStream_t stream);
// launch_gae, plus the map of every step (step_scen[T][N], from the episode-log records and the bound state's plane 4) and
// the per-map value-loss sums added into scores[n_scen + 1][3] (shipsim_gae_scored)
cudaError_t launch_gae_scored(const float *rew, const float *val, const unsigned char *done, int T, int N, float gamma, float lam, float *adv,
                              float *ret, const int4 *log_meta, const int *log_count, int log_cap, int call0, int steps_per_call,
                              const float4 *plane4, int n_scen, int *step_scen, double *scores, cudaStream_t stream);
cudaError_t launch_mlp_policy(const float *obs, int n, const float *w1, const float *b1, const float *w2, const float *b2, const float *w3,
                              const float *b3, const float *noise, float *out, long long *actions, cudaStream_t stream);
cudaError_t launch_render(const StepParams &p, int e, int img_w, int img_h, uint8_t *rgb, cudaStream_t stream);
// episode log, frames-only host path: the previous frame of the records of chunk [k0, k0 + kc) of call p.log_call
cudaError_t launch_log_prev_frames(const StepParams &p, const float4 *frames, const float4 *prev0, int k0, int kc, cudaStream_t stream);
cudaError_t launch_stats_reduce(double *slots, double *out, int clear, cudaStream_t stream);
// weighted scenario picks: table = [cdf: n_scen + 1][guide: n_scen + 1] built from the device array weights[n_scen]
cudaError_t launch_build_pick_table(const unsigned *weights, int n_scen, unsigned *table, cudaStream_t stream);

}  // namespace shipsim
