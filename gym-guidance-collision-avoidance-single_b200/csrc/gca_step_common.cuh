// gca_step_common.cuh - helpers of the step kernels in gca_step.cu (sm_100a).
#pragma once
#include <utility>

#include "gca_device.cuh"

namespace gca {

// bits of own_b.z (the ownship record the streaming pass reads)
constexpr uint32_t kOwnRuns = 1u;       // the reference's intruder loop runs for this env in this step
constexpr uint32_t kOwnPlane = 2u;      // parity of the env's current position plane

// Programmatic dependent launch: the kernels of a step are launched with programmatic stream serialization, so
// the next grid is staged (and its blocks scheduled as slots free up) while the current one drains.  A kernel
// calls pdl_wait() before it touches anything an earlier kernel of the stream wrote.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ownship state right after reset: (50, 50), min speed, heading pi/4 (PKG/SingleAircraftEnv.py:72-76), or with
// random_start random_pos(), random_speed(), random_heading() drawn in that order BEFORE the intruders
// (Simulators/SingleAircraftDiscrete9HEREnv.py:78-82); f32 position and velocity (Aircraft.__init__ :269-276)
template <bool TAPE>
__device__ __forceinline__ void reset_ownship(const gca_config& c, Draws<TAPE>& d, float2& pos, double2& hs, double2& vel) {
  double sn, cs;
  if (c.random_start) {
    double x, y, speed, heading;
    draw_pos(d, c, GCA_SLOT_OWN_RESET, GCA_BLOCK_POS, x, y);
    draw_speed_heading(d, c, GCA_SLOT_OWN_RESET, speed, heading);
    pos = make_float2((float)x, (float)y);
    hs = make_double2(heading, speed);
  } else {
    pos = make_float2(50.0f, 50.0f);
    hs = make_double2(3.141592653589793 / 4, c.min_speed);
  }
  gca_sincos(hs.x, &sn, &cs);
  vel = make_double2((double)(float)__dmul_rn(hs.y, cs), (double)(float)__dmul_rn(hs.y, sn));
}

template <bool TAPE>
__device__ __forceinline__ Draws<TAPE> make_draws(const StepArgs& a, size_t me, uint32_t tick) {
  Draws<TAPE> d;
  if constexpr (TAPE) {
    d.tape = a.tape + me * (size_t)a.tape_stride;
    d.cur = a.cursor[me];
  } else {
    d.k0 = a.key0; d.k1 = a.key1;
    d.env = a.env_id0 + (uint32_t)me;
    d.tick = tick;
  }
  return d;
}

// what _terminal_reward() returns when no intruder event outranks it: max steps / wall / goal / default
// (PKG/SingleAircraftEnv.py:173-183 and the variant rows of SURVEY.md 8(a))
struct Settled {
  double reward;
  int info;
  int done;
};
__device__ __forceinline__ Settled settle_own(const gca_config& c, const Derived& k, bool maxstep_hit, float2 pos, double2 goal) {
  double reward;
  int info, done = 0;
  if (maxstep_hit) {
    reward = 0.0; done = 1; info = GCA_INFO_MAXSTEPS;
  } else if (c.wall_kind != GCA_WALL_NONE && !in_map_f32(k, pos.x, pos.y)) {
    reward = c.r_wall; done = c.wall_kind == GCA_WALL_TERMINAL; info = GCA_INFO_WALL;
  } else {
    const double dg = dist_f64((double)pos.x, (double)pos.y, goal.x, goal.y);
    if (dg < c.goal_radius) {
      reward = c.r_goal; done = 1; info = GCA_INFO_GOAL;
    } else {
      reward = c.shaped_default ? ddiv_prepared(k, -dg, k.dv_shape, k.rc_shape) : c.r_default;
      info = GCA_INFO_NONE;
    }
  }
  return Settled{reward, info, done};
}

__device__ __forceinline__ void st_release_quad(float* p, float x, float y, float z, float w) {
  asm volatile("st.volatile.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ float4 ld_volatile_f4(const float4* p) {
  float4 v;
  asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}

// launch with programmatic stream serialization (see pdl_wait above)
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned blocks, unsigned threads, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

}  // namespace gca
