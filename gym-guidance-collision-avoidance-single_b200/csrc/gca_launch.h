// gca_launch.h - host-callable launchers of the kernels, and the host helpers they share.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <limits>

#include "gca_device.cuh"

namespace gca {
// smallest s with sqrt(s) >= thr, i.e. (sqrt(s) < thr) == (s < X); T = float or double
template <typename T>
T sq_threshold(T thr) {
  if (!(thr > 0)) return 0;
  T c = thr * thr;
  const T inf = std::numeric_limits<T>::infinity();
  while (c > 0 && std::sqrt(c) >= thr) c = std::nextafter(c, (T)0);
  while (std::sqrt(c) < thr) c = std::nextafter(c, inf);
  return c;
}


cudaError_t launch_step(bool faith, bool tape, const StepArgs& a, cudaStream_t st, cudaEvent_t* ev);
int step_launch_count(bool tape, int n_intruders, int obs_kind, bool turns);
cudaError_t launch_reset(bool faith, bool tape, const StepArgs& a, cudaStream_t st);
cudaError_t launch_observe(bool faith, const StepArgs& a, cudaStream_t st);
cudaError_t launch_compute_reward(const void* ag, long long n_ag, const void* g, long long m, double radius, int kind,
                                  int is_f64, float* out, cudaStream_t st);
cudaError_t launch_input_reward(const void* rows, long long m, int dim, int is_f64, const gca_input_reward_cfg* cfg,
                                double* out, uint8_t* done, cudaStream_t st);
cudaError_t launch_mcts_playouts(const gca_mcts_config* cfg, int n, const double* roots, long long n_roots, int playouts,
                                 int depth, const int8_t* first_action, uint64_t seed, uint32_t root_id0,
                                 double* rewards, int8_t* first_out, uint8_t* flags, cudaStream_t st);
cudaError_t launch_mcts_move(const gca_mcts_config* cfg, int n, double* states, const int32_t* actions, uint8_t* flags,
                             long long m, const double* tape, long long tape_stride, long long* cursor, uint64_t seed,
                             uint32_t id0, int first_frame, cudaStream_t st);
size_t mcts_search_workspace_bytes(const gca_mcts_config* cfg, int n, long long n_roots, int sims, int depth);
cudaError_t launch_mcts_search(const gca_mcts_config* cfg, int n, const double* roots, long long n_roots, int sims,
                               int depth, uint64_t seed, uint32_t root_id0, void* workspace, int32_t* best_action,
                               double* child_n, double* child_q, int32_t* child_action, cudaStream_t st);
cudaError_t launch_monitor_update(const void* reward, int is_f64, const uint8_t* done, long long n, float* ep_return,
                                  int32_t* ep_length, gca_episode_record* ring, long long cap, unsigned long long* count,
                                  uint32_t step, cudaStream_t st);
cudaError_t launch_stats_update(const uint8_t* done, const uint8_t* info, long long n, unsigned long long* stats,
                                cudaStream_t st);
cudaError_t launch_her_sample(const gca_her_episodes* ep, long long E, int T, int dim_o, int dim_u, int dim_g, int is_f64,
                              long long batch, double future_p, double radius, int kind, const gca_her_draws* dr,
                              uint64_t seed, uint32_t call, const gca_her_transitions* out, cudaStream_t st);
constexpr size_t kRasterSmemMax = 227 * 1024;   // dynamic shared memory one block may use
size_t raster_smem_bytes(int ow, int oh);        // what raster_kernel needs for an ow x oh output plane
cudaError_t launch_raster(const DevState& s, bool faithful, int W, int H, const uint8_t* sprites, uint8_t* frames,
                          long long env_stride, long long plane_stride, int n_planes, int slot,
                          const uint8_t* clear_mask, cudaStream_t st);
}  // namespace gca
