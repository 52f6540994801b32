// gca_her.cu - HER "future" relabelling sampler on a device-resident episode buffer (sm_100a).
//
// Reference: Algorithms/baselines-master/baselines/her/her_sampler.py:19-61 (_sample_her_transitions) as called by
// replay_buffer.py:sample (o_2 = o[:, 1:], ag_2 = ag[:, 1:]); reward_fun = the env's compute_reward
// (PKG/SingleAircraftHEREnv.py:194-196, PKG/SingleAircraftDiscreteHEREnv.py:184-186).
// One warp per sampled transition: the four draws are resolved (tape or Philox), then six rows are gathered with the
// widest vector width their alignment allows.  o[e][t] and o[e][t+1] are adjacent in memory.  Pure data movement:
// 2 * (2 dim_o + dim_u + 4 dim_g) * sizeof(REAL) + 16 bytes per transition, bound by HBM.
#include "gca_launch.h"

namespace gca {

struct HerArgs {
  const uint8_t *o, *u, *g, *ag;
  long long E, batch;
  int T, dim_o, dim_u, dim_g;
  double future_p, radius;
  int kind;
  const long long *episode_idxs, *t_samples;
  const double *u_her, *u_off;
  uint32_t key0, key1, call;
  uint8_t *out_o, *out_u, *out_g, *out_ag, *out_o2, *out_ag2;
  float* out_r;
  int32_t *out_e, *out_t, *out_ft;
};

// rows o[e][t] and o[e][t+1] (adjacent in memory) -> out_o[b], out_o2[b]: n vectors of type V per row, 4 + 4
// independent loads in flight per lane; streaming loads / stores (a row is touched once per sample)
template <typename V>
__device__ __forceinline__ void copy_row_pair(V* __restrict__ d0, V* __restrict__ d1, const V* __restrict__ s0, int n, int lane) {
  const V* s1 = s0 + n;
  for (int base = 0; base < n; base += 128) {
    V v0[4], v1[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = base + k * 32 + lane;
      if (i < n) { v0[k] = __ldcs(s0 + i); v1[k] = __ldcs(s1 + i); }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = base + k * 32 + lane;
      if (i < n) { __stcs(d0 + i, v0[k]); __stcs(d1 + i, v1[k]); }
    }
  }
}

// short rows (actions, goals): 4-byte words
__device__ __forceinline__ void copy_words(uint8_t* dst, const uint8_t* src, int nbytes, int lane) {
  for (int i = lane; i < nbytes / 4; i += 32) reinterpret_cast<uint32_t*>(dst)[i] = reinterpret_cast<const uint32_t*>(src)[i];
}

constexpr int kHerMinBlocks = 3;                  // blocks per SM (80 registers): 7 % more transitions/s than 2, 4 and 6 spill
template <typename R>
__global__ void __launch_bounds__(256, kHerMinBlocks) her_sample_kernel(const HerArgs a) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  const size_t ro = (size_t)a.dim_o * sizeof(R), ru = (size_t)a.dim_u * sizeof(R), rg = (size_t)a.dim_g * sizeof(R);
  // every o row starts at a multiple of ro from its base: one vector width for the whole launch
  const uintptr_t al = reinterpret_cast<uintptr_t>(a.o) | reinterpret_cast<uintptr_t>(a.out_o) |
                       reinterpret_cast<uintptr_t>(a.out_o2) | (uintptr_t)ro;
  const int vw = (al & 15) == 0 ? 16 : ((al & 7) == 0 ? 8 : 4);
  for (long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); b < a.batch; b += warps) {
    long long e;
    int t;
    double uh, uo;
    if (a.episode_idxs) {
      e = a.episode_idxs[b]; t = (int)a.t_samples[b]; uh = a.u_her[b]; uo = a.u_off[b];
    } else {
      const uint4 w0 = philox4x32_10(make_uint4((uint32_t)b, (uint32_t)(b >> 32), a.call, 0u), a.key0, a.key1);
      const uint4 w1 = philox4x32_10(make_uint4((uint32_t)b, (uint32_t)(b >> 32), a.call, 1u), a.key0, a.key1);
      e = (long long)__dmul_rn(u53(w0.x, w0.y), (double)a.E);
      t = (int)__dmul_rn(u53(w0.z, w0.w), (double)a.T);
      if (e > a.E - 1) e = a.E - 1;
      if (t > a.T - 1) t = a.T - 1;
      uh = u53(w1.x, w1.y); uo = u53(w1.z, w1.w);
    }
    const bool her = uh < a.future_p;                                  // her_indexes :33
    const int off = (int)__dmul_rn(uo, (double)(a.T - t));              // (uniform * (T - t_samples)).astype(int) :34-35
    const int ft = t + 1 + off;                                         // :36
    const size_t row_t = (size_t)e * (a.T + 1) + t;                     // o / ag have T + 1 rows per episode
    const size_t row_u = (size_t)e * a.T + t;
    uint8_t* d0 = a.out_o + (size_t)b * ro;
    uint8_t* d1 = a.out_o2 + (size_t)b * ro;
    const uint8_t* s0 = a.o + row_t * ro;
    if (vw == 16) copy_row_pair(reinterpret_cast<uint4*>(d0), reinterpret_cast<uint4*>(d1), reinterpret_cast<const uint4*>(s0), (int)(ro / 16), lane);
    else if (vw == 8) copy_row_pair(reinterpret_cast<uint2*>(d0), reinterpret_cast<uint2*>(d1), reinterpret_cast<const uint2*>(s0), (int)(ro / 8), lane);
    else copy_row_pair(reinterpret_cast<uint32_t*>(d0), reinterpret_cast<uint32_t*>(d1), reinterpret_cast<const uint32_t*>(s0), (int)(ro / 4), lane);
    copy_words(a.out_u + (size_t)b * ru, a.u + row_u * ru, (int)ru, lane);
    copy_words(a.out_ag + (size_t)b * rg, a.ag + row_t * rg, (int)rg, lane);
    copy_words(a.out_ag2 + (size_t)b * rg, a.ag + (row_t + 1) * rg, (int)rg, lane);
    // transitions['g'][her_indexes] = episode_batch['ag'][episode_idxs[her_indexes], future_t]  :41-42
    const uint8_t* gsrc = her ? a.ag + ((size_t)e * (a.T + 1) + ft) * rg : a.g + row_u * rg;
    copy_words(a.out_g + (size_t)b * rg, gsrc, (int)rg, lane);
    if (lane == 0) {
      // reward_fun(ag_2, g, info) :51-54 = compute_reward (gca_reward.cu), goals are 2-D
      const R* p = reinterpret_cast<const R*>(a.ag + (row_t + 1) * rg);
      const R* q = reinterpret_cast<const R*>(gsrc);
      bool gt, lt;
      if constexpr (sizeof(R) == 8) {
        const double dx = __dadd_rn(p[0], -q[0]), dy = __dadd_rn(p[1], -q[1]);
        const double d = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
        gt = d > a.radius; lt = d < a.radius;
      } else {
        const float dx = __fadd_rn(p[0], -q[0]), dy = __fadd_rn(p[1], -q[1]);
        const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        gt = d > (float)a.radius; lt = d < (float)a.radius;
      }
      reinterpret_cast<uint32_t*>(a.out_r)[b] = relabel_reward_bits(a.kind, gt, lt);
      if (a.out_e) a.out_e[b] = (int32_t)e;
      if (a.out_t) a.out_t[b] = t;
      if (a.out_ft) a.out_ft[b] = her ? ft : -1;
    }
  }
}

cudaError_t launch_her_sample(const gca_her_episodes* ep, long long E, int T, int dim_o, int dim_u, int dim_g, int is_f64,
                              long long batch, double future_p, double radius, int kind, const gca_her_draws* dr,
                              uint64_t seed, uint32_t call, const gca_her_transitions* out, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  HerArgs a{};
  a.o = (const uint8_t*)ep->o; a.u = (const uint8_t*)ep->u; a.g = (const uint8_t*)ep->g; a.ag = (const uint8_t*)ep->ag;
  a.E = E; a.batch = batch; a.T = T; a.dim_o = dim_o; a.dim_u = dim_u; a.dim_g = dim_g;
  a.future_p = future_p; a.radius = radius; a.kind = kind;
  if (dr) {
    a.episode_idxs = (const long long*)dr->episode_idxs; a.t_samples = (const long long*)dr->t_samples;
    a.u_her = dr->u_her; a.u_off = dr->u_offset;
  }
  a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.call = call;
  a.out_o = (uint8_t*)out->o; a.out_u = (uint8_t*)out->u; a.out_g = (uint8_t*)out->g; a.out_ag = (uint8_t*)out->ag;
  a.out_o2 = (uint8_t*)out->o_2; a.out_ag2 = (uint8_t*)out->ag_2; a.out_r = out->r;
  a.out_e = out->episode; a.out_t = out->t; a.out_ft = out->future_t;
  long long blocks = (batch + 7) / 8;
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (is_f64) her_sample_kernel<double><<<(unsigned)blocks, 256, 0, st>>>(a);
  else her_sample_kernel<float><<<(unsigned)blocks, 256, 0, st>>>(a);
  return cudaGetLastError();
}

}  // namespace gca
