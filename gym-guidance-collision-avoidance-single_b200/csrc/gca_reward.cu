// gca_reward.cu - HER relabelling reward (SURVEY a11), one thread per (achieved, desired) pair.
//   PKG/SingleAircraftHEREnv.py:194-196          -(norm(ag - g) > goal_radius).astype(f32)
//   PKG/SingleAircraftDiscreteHEREnv.py:184-186   (norm(ag - g) < goal_radius).astype(f32)
// np.linalg.norm(x, axis=-1) = sqrt(add.reduce(x*x)): plain multiply / add, in the input dtype.
// 20 bytes per pair (f32) or 36 (f64): purely HBM-bound, 16-byte loads, grid-stride.
#include "gca_launch.h"
#include "gca_step_common.cuh"

namespace gca {

template <typename T, typename T2>
__global__ void __launch_bounds__(256) reward_kernel(const T2* __restrict__ ag, long long n_ag, const T2* __restrict__ g,
                                                     long long m, double radius, int kind, float* __restrict__ out) {
  // launched with programmatic stream serialization: staged while the step's last kernel drains, and the next step's
  // first kernel is staged while this one runs (a plain launch between two steps cost ~2 us at each boundary)
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    const T2 a = ag[n_ag == m ? i : i % n_ag], b = g[i];     // (n_ag < m: the achieved goals repeat, k substitute goals each)
    bool gt, lt;
    if constexpr (sizeof(T) == 8) {
      const double dx = __dadd_rn(a.x, -b.x), dy = __dadd_rn(a.y, -b.y);
      const double d = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
      gt = d > radius;
      lt = d < radius;
    } else {
      const float dx = __fadd_rn(a.x, -b.x), dy = __fadd_rn(a.y, -b.y);
      const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
      gt = d > (float)radius;
      lt = d < (float)radius;
    }
    reinterpret_cast<uint32_t*>(out)[i] = relabel_reward_bits(kind, gt, lt);
  }
}

cudaError_t launch_compute_reward(const void* ag, long long n_ag, const void* g, long long m, double radius, int kind,
                                  int is_f64, float* out, cudaStream_t st) {
  if (m <= 0) return cudaSuccess;
  long long blocks = (m + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (is_f64)
    return launch_pdl(reward_kernel<double, double2>, (unsigned)blocks, 256, st, (const double2*)ag, n_ag, (const double2*)g,
                      m, radius, kind, out);
  return launch_pdl(reward_kernel<float, float2>, (unsigned)blocks, 256, st, (const float2*)ag, n_ag, (const float2*)g, m,
                    radius, kind, out);
}

// compute_input_reward(new_inputs) of Simulators/SingleAircraftDiscrete9HEREnv.py:244-276 for m relabelled
// (observation + goal) rows at once: thread = row.  The reference's arithmetic, statement by statement: the
// un-normalisation products and metric()'s differences / squares in the dtype of the row (NumPy scalars), the square
// root in f64 (math.sqrt), the listed intruders read with stride 4 although each has 5 entries (idx * 4 + 4: kept),
// the first listed intruder inside minimum_separation decides (conflict, or NMAC inside NMAC_dist), then goal /
// step penalty / shaped default.  done = (r == 10 or r == -10), the literals of Algorithms/pytorch/agent_her.py:117.
template <typename T>
__global__ void __launch_bounds__(256) input_reward_kernel(const T* __restrict__ rows, long long m, int dim,
                                                           const gca_input_reward_cfg c, double* __restrict__ out,
                                                           uint8_t* __restrict__ done) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const T* v = rows + i * (long long)dim;
  const T w = (T)c.window_width, h = (T)c.window_height;   // (a Python number: it takes the array scalar's dtype)
  auto metric = [](T x1, T y1, T x2, T y2) {
    const T dx = x1 - x2, dy = y1 - y2;                    // (-fmad=false: single multiplies and adds)
    return sqrt((double)(dx * dx + dy * dy));
  };
  const T ownx = v[0] * w, owny = v[1] * h, gx = v[dim - 2] * w, gy = v[dim - 1] * h;
  const double dist_goal = metric(ownx, owny, gx, gy);
  double r;
  bool settled = false;
  if (c.has_intruders) {
    for (int idx = 0; idx < c.n_listed && !settled; ++idx) {
      const T ix = v[idx * 4 + 4] * w, iy = v[idx * 4 + 5] * h;
      const double d = metric(ownx, owny, ix, iy);
      if (d < c.minimum_separation) {
        r = d < c.nmac_dist ? c.nmac_penalty : c.conflict_penalty;
        settled = true;
      }
    }
  }
  if (!settled) {
    if (dist_goal < c.goal_radius) r = c.goal_reward;
    else r = c.sparse_reward ? c.step_penalty : -dist_goal / 1200.0;
  }
  out[i] = r;
  if (done) done[i] = (r == 10.0 || r == -10.0) ? 1 : 0;
}

cudaError_t launch_input_reward(const void* rows, long long m, int dim, int is_f64, const gca_input_reward_cfg* cfg,
                                double* out, uint8_t* done, cudaStream_t st) {
  if (m <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((m + 255) / 256);
  if (is_f64) input_reward_kernel<double><<<blocks, 256, 0, st>>>((const double*)rows, m, dim, *cfg, out, done);
  else input_reward_kernel<float><<<blocks, 256, 0, st>>>((const float*)rows, m, dim, *cfg, out, done);
  return cudaGetLastError();
}

// VecMonitor.step_wait (baselines common/vec_env/vec_monitor.py:21-37) for the whole batch: thread = env.  Finished
// episodes are appended to a device ring (warp-aggregated slot reservation: one atomic per warp).
template <typename R>
__global__ void __launch_bounds__(256) monitor_kernel(const R* __restrict__ reward, const uint8_t* __restrict__ done,
                                                      long long n, float* __restrict__ ep_return,
                                                      int32_t* __restrict__ ep_length, gca_episode_record* __restrict__ ring,
                                                      long long cap, unsigned long long* __restrict__ count, uint32_t step) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < n;
  float ret = 0.0f;
  int len = 0;
  bool fin = false;
  if (valid) {
    ret = __fadd_rn(ep_return[i], (float)reward[i]);       // self.eprets += rews  (float32)
    len = ep_length[i] + 1;                                // self.eplens += 1
    fin = done[i] != 0;
    ep_return[i] = fin ? 0.0f : ret;
    ep_length[i] = fin ? 0 : len;
  }
  const unsigned m = __ballot_sync(0xffffffffu, fin);
  if (m) {
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == __ffs(m) - 1) base = atomicAdd(count, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (fin) {
      gca_episode_record rec;
      rec.env = (int32_t)i; rec.length = len; rec.ep_return = ret; rec.step = step;
      ring[(base + __popc(m & ((1u << lane) - 1u))) % (unsigned long long)cap] = rec;
    }
  }
}

cudaError_t launch_monitor_update(const void* reward, int is_f64, const uint8_t* done, long long n, float* ep_return,
                                  int32_t* ep_length, gca_episode_record* ring, long long cap, unsigned long long* count,
                                  uint32_t step, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (is_f64) monitor_kernel<double><<<blocks, 256, 0, st>>>((const double*)reward, done, n, ep_return, ep_length, ring, cap, count, step);
  else monitor_kernel<float><<<blocks, 256, 0, st>>>((const float*)reward, done, n, ep_return, ep_length, ring, cap, count, step);
  return cudaGetLastError();
}

// step / episode / outcome counters of one step, thread = env, one atomic per warp and non-zero counter
__global__ void __launch_bounds__(256) stats_kernel(const uint8_t* __restrict__ done, const uint8_t* __restrict__ info,
                                                    long long n, unsigned long long* __restrict__ stats) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < n;
  const int code = valid ? info[i] : -1;
  const bool fin = valid && done[i] != 0;
  const int lane = threadIdx.x & 31;
  const unsigned counts[7] = {
      (unsigned)__popc(__ballot_sync(0xffffffffu, valid)), (unsigned)__popc(__ballot_sync(0xffffffffu, fin)),
      (unsigned)__popc(__ballot_sync(0xffffffffu, code == GCA_INFO_NMAC)),
      (unsigned)__popc(__ballot_sync(0xffffffffu, code == GCA_INFO_CONFLICT)),
      (unsigned)__popc(__ballot_sync(0xffffffffu, code == GCA_INFO_GOAL)),
      (unsigned)__popc(__ballot_sync(0xffffffffu, code == GCA_INFO_WALL)),
      (unsigned)__popc(__ballot_sync(0xffffffffu, code == GCA_INFO_MAXSTEPS))};
  if (lane < 7 && counts[lane]) atomicAdd(&stats[lane], (unsigned long long)counts[lane]);
}

cudaError_t launch_stats_update(const uint8_t* done, const uint8_t* info, long long n, unsigned long long* stats,
                                cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  stats_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(done, info, n, stats);
  return cudaGetLastError();
}

}  // namespace gca
