// gca_device.cuh - device-side building blocks of the step hot path (sm_100a).
//
// Compiled with -fmad=false: every arithmetic operation that has to reproduce the reference's
// NumPy scalar rounding is written with an explicit round-to-nearest intrinsic, and the one
// place where the reference (through OpenBLAS ddot) fuses is an explicit __fma_rn.
// Citations: PKG = gym_guidance_collision_avoidance_single/envs of the reference tree.
#pragma once
#include <math_constants.h>

#include <cuda_runtime.h>
#include <stdint.h>

#include "gca.h"
#include "gca_math.h"

namespace gca {

// ------------------------------------------------------------------------------ device state
// Everything is laid out for "lane = env": a warp works on a tile of 32 consecutive envs and lane e
// of the warp touches env 32*t + e only.
//   per-env scalars   SoA by field, [B]: one coalesced access per warp.
//   intruder planes   tile-planar: for tile t and 16-byte unit u the 32 lanes' units are adjacent,
//                         plane[(t * units + u) * 32 + e]            (512 bytes per (t, u))
//       pos  FAST     unit u = float4 (x, y) of intruders 2u, 2u+1           units = U = ceil(N/2)
//            FAITHFUL unit i = double2 (x, y) of intruder i (an f32 value unless flagged)  units = 2U
//       vel           unit u = float4 (vx, vy) of intruders 2u, 2u+1         units = U
//       conflict / f64 flag words and the per-step event words: word w of env e at words[(t * Wd + w) * 32 + e]
//   so every warp-wide 16-byte access is one contiguous 512-byte line and any run of units of a tile is
//   one contiguous block.
// Positions are double-buffered (two planes).  The plane that holds env e's current positions is
// tick(e) & 1; a step reads it, writes the other one and increments the tick.  The intruder pass of a
// step therefore never overwrites its input, which makes it order-free: any warp can advance any 8
// intruders of any tile at any time, and the rare "the reference's loop returned at intruder i"
// case (NMAC, Q9) is repaired afterwards from the untouched old plane.
// bit i%32 of conflict word i/32 = Aircraft.conflict of intruder i; the f64 words flag positions
// whose dtype became f64 after a retried spawn (Q3).
struct DevState {
  float2* own_pos;        // [B]
  double2* own_hs;        // [B]   (heading, speed)
  double2* own_vel;       // [B]
  uint8_t* own_vel_f32;   // [B]
  double2* goal;          // [B]
  int4* counters;         // [B]   (no_conflict, ep_steps, tick, episodes)
  uint8_t* ipos;          // [2][T][U or 2U][32] 16-byte units
  uint8_t* ivel;          // [T][U][32] float4
  uint32_t* cflag;        // [T][Wd][32]
  uint32_t* dflag;        // [T][Wd][32]  (FAITHFUL)
  double2* ihs;           // [T][N][32] (heading, speed) of every intruder - only handles whose intruders turn or whose
                          // observation shows them keep it (Simulators/SingleAircraftMCTSRandIntruderEnv.py), else nullptr
  // hand-over between the three kernels of a step
  float4* own_b;          // [T*32] (own x, own y, bits: 1 = the intruder loop runs, 2 = plane parity, -)
  uint32_t* ev_conf;      // [T][Wd][32] bit i: intruder i is inside the separation radius after its advance
  uint32_t* ev_gone;      // [T][Wd][32] bit i: intruder i left the map
  int* ev_nmac;           // [T*32] lowest intruder index inside the NMAC radius (INT_MAX: none)
  uint32_t* ev_near;      // [T*32] shaped_nearest, FAST: bits of the smallest squared ownship-intruder distance of the step
  uint64_t align_pad;     // unused: see StepArgs::align_pad
  // PHILOX handles (two kernels per step, see gca_step.cu)
  double2* pre;           // [T*32] what the ownship role settled before the intruders were looked at: (reward candidate,
                          //        bits: info | done << 8) of wall / goal / default / max-steps - the finish takes it unless an
                          //        intruder event outranks it
  uint32_t* step_seq;     // [1] steps launched on this handle; own_b.w of step k carries stamp k + 1 (valid under graph replay)
  int* error_flag;        // [1] 1: a streaming lane's ownship record never arrived (dispatch order broke)
  size_t pos_plane;       // bytes of one position plane
  int B, N, T, U, W, Wd;
};

template <bool FAITH>
struct pos2 { using type = float2; };
template <>
struct pos2<true> { using type = double2; };

__host__ __device__ inline void plane_layout(DevState& s, bool faithful) {
  s.T = (s.B + 31) / 32;
  s.U = (s.N + 1) / 2;
  s.W = (s.N + 31) / 32;
  s.Wd = s.W > 0 ? s.W : 1;
  s.pos_plane = (size_t)s.T * (size_t)(s.U > 0 ? s.U : 1) * 512u * (faithful ? 2u : 1u);
}
__host__ __device__ inline size_t vel_plane_bytes(const DevState& s) { return (size_t)s.T * (size_t)(s.U > 0 ? s.U : 1) * 512u; }
__host__ __device__ inline size_t flag_plane_words(const DevState& s) { return (size_t)s.T * (size_t)s.Wd * 32u; }

// byte offsets of intruder i of env `env` inside a position plane / the velocity plane
__host__ __device__ inline size_t ipos_offset(const DevState& s, bool faithful, size_t env, int i) {
  const size_t t = env >> 5, e = env & 31;
  if (faithful) return ((t * (size_t)(2 * s.U) + (size_t)i) * 32 + e) * 16;
  return ((t * (size_t)s.U + (size_t)(i >> 1)) * 32 + e) * 16 + (size_t)(i & 1) * 8;
}
__host__ __device__ inline size_t ivel_offset(const DevState& s, size_t env, int i) {
  const size_t t = env >> 5, e = env & 31;
  return ((t * (size_t)s.U + (size_t)(i >> 1)) * 32 + e) * 16 + (size_t)(i & 1) * 8;
}
__host__ __device__ inline size_t ihs_index(const DevState& s, size_t env, int i) {
  const size_t t = env >> 5, e = env & 31;
  return (t * (size_t)s.N + (size_t)i) * 32 + e;
}
__host__ __device__ inline size_t flag_index(const DevState& s, size_t env, int w) {
  const size_t t = env >> 5, e = env & 31;
  return (t * (size_t)s.Wd + (size_t)w) * 32 + e;
}

// Constants derived from gca_config on the host (gca_abi.cu), exact by construction.
// `d < thr` on a correctly rounded sqrt is monotone in its argument, so each distance test is
// done on the squared distance against X = min{ s : sqrt(s) >= thr } - same truth value, no sqrt.
struct Derived {
  float sep2_f, nmac2_f, init2_f;     // f32 distances (thr taken as f32, NumPy 2 weak scalars)
  double sep2_d, nmac2_d, init2_d;    // f64 distances
  double goal2_d;                     // goal_radius, for the squared f64 ownship-goal distance (dist2_f64)
  float win_w, win_h;                 // Box bounds are f32 (PKG/SingleAircraftEnv.py:38-41)
  float ob_w, ob_h, inv_ob_w, inv_ob_h;   // x / Config.window_* in f32, and RN(1/.) for gca_div_const_f32
  float ms, den, inv_den;             // normalize_velocity: (v + ms) / den in f32
  int div1_ok;                        // the one-correction division is exact for ob_w, ob_h and den
  // f64 divisors of the observation tail / shaped reward and their correctly rounded reciprocals (gca_div_const_f64)
  double dv_w, dv_h, dv_speed, dv_2pi, dv_vel, dv_shape;       // window w/h, max-min speed, 2*pi, 2*max_speed, 1200
  double rc_w, rc_h, rc_speed, rc_2pi, rc_vel, rc_shape;
  int ddiv_ok;                        // all six divisors qualify (gca_div_f64_divisor_ok)
  float drift_f;                      // f32(position_drift), added to the f32 velocity of every advance
  int has_drift;                      // position_drift != 0
  // u53(...) < turn_prob on the 53-bit integer: v * 2^-53 < t  <=>  v < ceil(t * 2^53) (both sides exact)
  unsigned long long turn_thresh;
};

// x / d in f64, correctly rounded, for the host-prepared divisors of Derived
__device__ __forceinline__ double ddiv_prepared(const Derived& k, double x, double d, double inv_d) {
  return k.ddiv_ok ? gca_div_const_f64(x, d, inv_d) : __ddiv_rn(x, d);
}

// x / d in f32, correctly rounded, for the host-prepared divisors of Derived
__device__ __forceinline__ float div_prepared(const Derived& k, float x, float d, float inv_d) {
  float q = __fmul_rn(x, inv_d);
  float r = __fmaf_rn(-q, d, x);
  q = __fmaf_rn(r, inv_d, q);
  if (!k.div1_ok) {                   // general divisor: second Markstein step (gca_div_const_f32)
    r = __fmaf_rn(-q, d, x);
    q = __fmaf_rn(r, inv_d, q);
  }
  return q;
}

struct StepArgs {
  DevState s;
  gca_config cfg;
  Derived k;
  const void* actions;
  const double* tape;
  long long tape_stride;
  long long* cursor;
  const uint8_t* mask;    // reset only
  uint32_t key0, key1, env_id0;
  int D;                  // observation row length
  int auto_reset;
  int own_blocks;         // PHILOX: leading blocks of step_intruders_kernel that play the ownship role (0: TAPE, own kernel)
  int align_pad;          // unused: with DevState::align_pad it keeps every field at the offset modulo 16 that the step
                          // kernels were tuned with - the compiler fetches a 16-byte aligned pair of 8-byte fields from
                          // the constant bank with one load, so shifting the fields by 8 bytes changes the kernels' code
  void* obs;
  void* achieved;
  void* desired;
  void* reward;
  uint8_t* done;
  uint8_t* info;
  void* nearest;          // REAL [B] or nullptr (shaped_nearest variants)
};

constexpr unsigned FULL = 0xffffffffu;

// ------------------------------------------------------------------------------ L2 eviction hints
// The streaming pass moves ~215 MB per step through a 126 MB L2; nothing of it is touched again before it would
// have been evicted anyway.  Marking that traffic evict_first keeps the ~10 MB that the other kernels of a step
// DO come back to (per-env scalars, event words, flag words) resident, so their dependent loads are L2 hits.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// The opposite hint for the few megabytes that a LATER kernel of the same step reads first (what the ownship role
// leaves for the finish: position, counters, reward candidate): evict_last keeps them in the L2
// across the 200 MB stream, so the finish kernel's first loads are L2 hits instead of DRAM round trips.
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float4 ldg_stream(const void* ptr, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(ptr), "l"(pol));
  return v;
}
__device__ __forceinline__ void stg_stream2(void* ptr, float x, float y, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(ptr), "f"(x), "f"(y), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_stream(void* ptr, const float4& v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(ptr), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w), "l"(pol)
               : "memory");
}

// ------------------------------------------------------------------------------ Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  const unsigned long long v = ((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6);
  return __dmul_rn((double)v, 1.0 / 9007199254740992.0);
}

// ------------------------------------------------------------------------------ draw sources
// A Draws object belongs to one env.  TAPE: values recorded from the reference's global numpy
// stream, consumed in the reference's order.  PHILOX: counter = (env id, tick, slot, block).
template <bool TAPE>
struct Draws;

template <>
struct Draws<true> {
  const double* tape;
  long long cur;
  __device__ __forceinline__ double next() { return tape[cur++]; }
};

template <>
struct Draws<false> {
  uint32_t k0, k1, env, tick;
  __device__ __forceinline__ void uniform2(uint32_t slot, uint32_t block, double& u0, double& u1) const {
    const uint4 w = philox4x32_10(make_uint4(env, tick, slot, block), k0, k1);
    u0 = u53(w.x, w.y);
    u1 = u53(w.z, w.w);
  }
};

// np.random.uniform(low=[0,0], high=[W,H])   PKG/SingleAircraftEnv.py:240-244
template <bool TAPE>
__device__ __forceinline__ void draw_pos(Draws<TAPE>& d, const gca_config& c, uint32_t slot, uint32_t block,
                                         double& x, double& y) {
  if constexpr (TAPE) {
    x = d.next();
    y = d.next();
  } else {
    double u0, u1;
    d.uniform2(slot, block, u0, u1);
    x = __dadd_rn(0.0, __dmul_rn(__dadd_rn(c.window_width, -0.0), u0));   // low + (high - low) * u
    y = __dadd_rn(0.0, __dmul_rn(__dadd_rn(c.window_height, -0.0), u1));
  }
}

// Goal(random_pos()) :93, or random_goal_pos() = uniform(low=[m, m], high=[W - m, H - m]) with goal_margin m
// (Simulators/SingleAircraftDiscrete3HEREnv.py:349-353)
template <bool TAPE>
__device__ __forceinline__ void draw_goal(Draws<TAPE>& d, const gca_config& c, double& x, double& y) {
  if constexpr (!TAPE) {
    if (c.goal_margin > 0) {
      double u0, u1;
      d.uniform2(GCA_SLOT_GOAL, GCA_BLOCK_POS, u0, u1);
      const double m = c.goal_margin;
      x = __dadd_rn(m, __dmul_rn(__dadd_rn(__dadd_rn(c.window_width, -m), -m), u0));   // low + (high - low) * u
      y = __dadd_rn(m, __dmul_rn(__dadd_rn(__dadd_rn(c.window_height, -m), -m), u1));
      return;
    }
  }
  draw_pos(d, c, GCA_SLOT_GOAL, GCA_BLOCK_POS, x, y);
}

// random_speed(), random_heading()   PKG/SingleAircraftEnv.py:246-250
template <bool TAPE>
__device__ __forceinline__ void draw_speed_heading(Draws<TAPE>& d, const gca_config& c, uint32_t slot,
                                                   double& speed, double& heading) {
  if constexpr (TAPE) {
    speed = d.next();
    heading = d.next();
  } else {
    double u0, u1;
    d.uniform2(slot, GCA_BLOCK_SPEED_HEADING, u0, u1);
    speed = __dadd_rn(c.min_speed, __dmul_rn(__dadd_rn(c.max_speed, -c.min_speed), u0));
    heading = __dadd_rn(0.0, __dmul_rn(6.283185307179586, u1));
  }
}

// the two np.random.normal(0, sigma) calls of Ownship.step   PKG/SingleAircraftEnv.py:301,304
template <bool TAPE>
__device__ __forceinline__ void draw_own_noise(Draws<TAPE>& d, const gca_config& c, double& nh, double& ns) {
  if constexpr (TAPE) {
    nh = d.next();
    ns = d.next();
  } else {
    double u0, u1, sn, cs;
    d.uniform2(GCA_SLOT_OWNSHIP, 0u, u0, u1);
    const double r = __dsqrt_rn(__dmul_rn(-2.0, gca_log(__dadd_rn(1.0, -u0))));
    gca_sincos(__dmul_rn(6.283185307179586, u1), &sn, &cs);
    nh = __dadd_rn(0.0, __dmul_rn(c.heading_sigma, __dmul_rn(r, cs)));
    ns = __dadd_rn(0.0, __dmul_rn(c.speed_sigma, __dmul_rn(r, sn)));
  }
}

// ------------------------------------------------------------------------------ distances
// dist(): np.linalg.norm(p1 - p2)   PKG/SingleAircraftEnv.py:312-313 (SURVEY a6)
//   f32 - f32 : sqrtf(fl(fl(dx*dx) + fl(dy*dy)))         (OpenBLAS sdot, no FMA)
//   with f64  : sqrt(fma(dy, dy, fl(dx*dx)))             (OpenBLAS ddot tail)
__device__ __forceinline__ float dist2_f32(float ax, float ay, float bx, float by) {
  const float dx = __fadd_rn(ax, -bx), dy = __fadd_rn(ay, -by);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}
__device__ __forceinline__ double dist2_f64(double ax, double ay, double bx, double by) {
  const double dx = __dadd_rn(ax, -bx), dy = __dadd_rn(ay, -by);
  return __fma_rn(dy, dy, __dmul_rn(dx, dx));
}
__device__ __forceinline__ double dist_f64(double ax, double ay, double bx, double by) {
  return __dsqrt_rn(dist2_f64(ax, ay, bx, by));
}

// position_range.contains(p): inclusive, f32 bounds   PKG/SingleAircraftEnv.py:38-41,153
__device__ __forceinline__ bool in_map_f32(const Derived& k, float x, float y) {
  return x >= 0.0f && y >= 0.0f && x <= k.win_w && y <= k.win_h;
}
__device__ __forceinline__ bool in_map_f64(const Derived& k, double x, double y) {
  return x >= 0.0 && y >= 0.0 && x <= (double)k.win_w && y <= (double)k.win_h;
}

// ------------------------------------------------------------------------------ intruder record
// FAST: everything f32.  FAITHFUL: the position is a double that holds either an f32 value
// (is64 == false) or a true f64 (a spawn that was retried, Q3).
template <bool FAITH>
struct Intr {
  float px, py, vx, vy;
  static constexpr bool is64 = false;
};
template <>
struct Intr<true> {
  double px, py;
  float vx, vy;
  bool is64;
};

// scattered (one intruder of one env) accessors of the global planes: reset, respawn, repair, observe, raster.
// `plane` = 0 / 1 selects the position buffer.
template <bool FAITH>
__device__ __forceinline__ void load_intruder(const DevState& s, int plane, size_t env, int i, Intr<FAITH>& it) {
  const uint8_t* base = s.ipos + (size_t)plane * s.pos_plane;
  if constexpr (FAITH) {
    const double2 p = *reinterpret_cast<const double2*>(base + ipos_offset(s, true, env, i));
    it.px = p.x;
    it.py = p.y;
    it.is64 = (s.dflag[flag_index(s, env, i >> 5)] >> (i & 31)) & 1u;
  } else {
    const float2 p = *reinterpret_cast<const float2*>(base + ipos_offset(s, false, env, i));
    it.px = p.x;
    it.py = p.y;
  }
  const float2 v = *reinterpret_cast<const float2*>(s.ivel + ivel_offset(s, env, i));
  it.vx = v.x;
  it.vy = v.y;
}

template <bool FAITH>
__device__ __forceinline__ void store_ipos(const DevState& s, int plane, size_t env, int i, const Intr<FAITH>& it) {
  uint8_t* base = s.ipos + (size_t)plane * s.pos_plane;
  if constexpr (FAITH) *reinterpret_cast<double2*>(base + ipos_offset(s, true, env, i)) = make_double2(it.px, it.py);
  else *reinterpret_cast<float2*>(base + ipos_offset(s, false, env, i)) = make_float2(it.px, it.py);
}

__device__ __forceinline__ void store_ivel(const DevState& s, size_t env, int i, float vx, float vy) {
  *reinterpret_cast<float2*>(s.ivel + ivel_offset(s, env, i)) = make_float2(vx, vy);
}

// where spawn() leaves the (heading, speed) of intruder i - nullptr for the handles that do not keep them
__device__ __forceinline__ double2* ihs_slot(const DevState& s, size_t env, int i) {
  return s.ihs ? s.ihs + ihs_index(s, env, i) : nullptr;
}

// intruder.position += intruder.velocity   PKG/SingleAircraftEnv.py:150, and the map test :153;
// `+= intruder.velocity + self.position_sigma` (f32 array + Python float: an f32 sum) with a position drift
// (Simulators/SingleAircraftMCTSRandIntruderEnv.py:183)
template <bool FAITH, bool DRIFT = false>
__device__ __forceinline__ bool advance(const Derived& k, Intr<FAITH>& it) {
  const float vx = DRIFT ? __fadd_rn(it.vx, k.drift_f) : it.vx;
  const float vy = DRIFT ? __fadd_rn(it.vy, k.drift_f) : it.vy;
  if constexpr (FAITH) {
    if (it.is64) {                                       // f64 + f32 -> f64
      it.px = __dadd_rn(it.px, (double)vx);
      it.py = __dadd_rn(it.py, (double)vy);
      return !in_map_f64(k, it.px, it.py);
    }
    const float fx = __fadd_rn((float)it.px, vx), fy = __fadd_rn((float)it.py, vy);
    it.px = (double)fx;
    it.py = (double)fy;
    return !in_map_f32(k, fx, fy);
  } else {
    it.px = __fadd_rn(it.px, vx);
    it.py = __fadd_rn(it.py, vy);
    return !in_map_f32(k, it.px, it.py);
  }
}

// ownship <-> intruder `dist < threshold` tests in the dtype the reference uses
template <bool FAITH>
__device__ __forceinline__ void separation(const Derived& k, float ox, float oy, const Intr<FAITH>& it, bool& lt_sep,
                                           bool& lt_nmac, bool& lt_init) {
  if constexpr (FAITH) {
    if (it.is64) {
      const double s2 = dist2_f64((double)ox, (double)oy, it.px, it.py);
      lt_sep = s2 < k.sep2_d;
      lt_nmac = s2 < k.nmac2_d;
      lt_init = s2 < k.init2_d;
      return;
    }
  }
  const float s2 = dist2_f32(ox, oy, (float)it.px, (float)it.py);
  lt_sep = s2 < k.sep2_f;
  lt_nmac = s2 < k.nmac2_f;
  lt_init = s2 < k.init2_f;
}

// Aircraft(random_pos(), random_speed(), random_heading()) + rejection loop
// PKG/SingleAircraftEnv.py:229-238,269-278 (reset: :80-88)
template <bool FAITH, bool TAPE>
__device__ __forceinline__ void spawn(Draws<TAPE>& d, const gca_config& c, const Derived& k, uint32_t slot, float ox,
                                      float oy, Intr<FAITH>& it, double2* hs_out) {
  double x, y, speed, heading, sn, cs;
  draw_pos(d, c, slot, GCA_BLOCK_POS, x, y);
  draw_speed_heading(d, c, slot, speed, heading);
  if (hs_out) *hs_out = make_double2(heading, speed);    // Aircraft.heading / .speed, kept by the turning-intruder variant
  it.px = (float)x;
  it.py = (float)y;
  if constexpr (FAITH) it.is64 = false;
  gca_sincos(heading, &sn, &cs);
  it.vx = (float)__dmul_rn(speed, cs);
  it.vy = (float)__dmul_rn(speed, sn);
  int retries = 0;
  for (;;) {
    bool a, b, lt_init;
    separation<FAITH>(k, ox, oy, it, a, b, lt_init);
    if (!lt_init) break;
    if (!TAPE && retries >= GCA_MAX_SPAWN_RETRIES) break;
    draw_pos(d, c, slot, GCA_BLOCK_RETRY0 + (uint32_t)retries, x, y);
    ++retries;
    if constexpr (FAITH) {       // intruder.position = self.random_pos(): a raw f64 array (Q3)
      it.px = x;
      it.py = y;
      it.is64 = true;
    } else {                     // FAST storage rule: rounded to f32
      it.px = (float)x;
      it.py = (float)y;
    }
  }
}

// ------------------------------------------------------------------------------ observation
template <bool FAITH>
using real_t = typename std::conditional<FAITH, double, float>::type;

__device__ __forceinline__ bool own_first(const gca_config& c) {
  return c.obs_kind == GCA_OBS_HER || c.obs_kind == GCA_OBS_DHER;
}

// normalize_velocity() on an f32 velocity   PKG/SingleAircraftEnv.py:104-106
__device__ __forceinline__ float norm_vel_f32(const Derived& k, float v) {
  return div_prepared(k, __fadd_rn(v, k.ms), k.den, k.inv_den);
}
__device__ __forceinline__ double norm_vel_f64(const gca_config& c, const Derived& k, double v) {
  return ddiv_prepared(k, __dadd_rn(v, c.max_speed), k.dv_vel, k.rc_vel);
}

// the four entries of an intruder   PKG/SingleAircraftEnv.py:108-114 (raw: Simulators/SingleAircraftMCTSEnv.py:107-112)
template <bool FAITH>
__device__ __forceinline__ void obs_intruder_entries(const StepArgs& a, const Intr<FAITH>& it, real_t<FAITH>& o0,
                                                     real_t<FAITH>& o1, real_t<FAITH>& o2, real_t<FAITH>& o3) {
  using R = real_t<FAITH>;
  const gca_config& c = a.cfg;
  const Derived& k = a.k;
  if (c.obs_kind == GCA_OBS_RAW) {
    o0 = (R)it.px; o1 = (R)it.py; o2 = (R)it.vx; o3 = (R)it.vy;
  } else {
    bool wide = false;
    if constexpr (FAITH) wide = it.is64;
    if (wide) {
      o0 = (R)ddiv_prepared(k, (double)it.px, k.dv_w, k.rc_w);
      o1 = (R)ddiv_prepared(k, (double)it.py, k.dv_h, k.rc_h);
    } else {
      o0 = (R)div_prepared(k, (float)it.px, k.ob_w, k.inv_ob_w);
      o1 = (R)div_prepared(k, (float)it.py, k.ob_h, k.inv_ob_h);
    }
    o2 = (R)norm_vel_f32(k, it.vx);
    o3 = (R)norm_vel_f32(k, it.vy);
  }
}

// the four entries of intruder i into its observation row; `base` points at the row's first intruder entry
template <bool FAITH>
__device__ __forceinline__ void write_obs_intruder(const StepArgs& a, real_t<FAITH>* base, int i,
                                                   const Intr<FAITH>& it) {
  using R = real_t<FAITH>;
  const gca_config& c = a.cfg;
  if (c.obs_kind == GCA_OBS_NONE || c.obs_kind == GCA_OBS_NEAREST || c.obs_kind == GCA_OBS_RAW6) return;   // (NEAREST: nearest_obs_kernel, RAW6: turn_obs_kernel)
  R o0, o1, o2, o3;
  obs_intruder_entries<FAITH>(a, it, o0, o1, o2, o3);
  R* p = base + 4 * (size_t)i;
  if constexpr (FAITH) {
    reinterpret_cast<double2*>(p)[0] = make_double2(o0, o1);
    reinterpret_cast<double2*>(p)[1] = make_double2(o2, o3);
  } else {
    if (!own_first(c)) {
      *reinterpret_cast<float4*>(p) = make_float4(o0, o1, o2, o3);
    } else {   // HER rows start at element 6: only 8-byte aligned
      reinterpret_cast<float2*>(p)[0] = make_float2(o0, o1);
      reinterpret_cast<float2*>(p)[1] = make_float2(o2, o3);
    }
  }
}

// The same four entries for the specialised hot path (FAST, GCA_OBS_VECTOR, one-correction
// division verified exact for all three divisors on the host): no run-time layout tests.
__device__ __forceinline__ float div_one(float x, float d, float inv_d) {
  const float q = __fmul_rn(x, inv_d);
  return __fmaf_rn(__fmaf_rn(-q, d, x), inv_d, q);
}
__device__ __forceinline__ float4 obs_intruder_vec(const Derived& k, float px, float py, float vx, float vy) {
  return make_float4(div_one(px, k.ob_w, k.inv_ob_w), div_one(py, k.ob_h, k.inv_ob_h),
                     div_one(__fadd_rn(vx, k.ms), k.den, k.inv_den), div_one(__fadd_rn(vy, k.ms), k.den, k.inv_den));
}

template <bool FAITH>
__device__ __forceinline__ real_t<FAITH>* obs_intruder_base(const StepArgs& a, size_t env) {
  return reinterpret_cast<real_t<FAITH>*>(a.obs) + env * (size_t)a.D + (own_first(a.cfg) ? 6 : 0);
}

// ownship entries, goal entries, achieved/desired   PKG/SingleAircraftEnv.py:115-124,
// PKG/SingleAircraftHEREnv.py:113-139, PKG/SingleAircraftDiscreteHEREnv.py:128-133
template <bool FAITH>
__device__ __forceinline__ void write_obs_own(const StepArgs& a, size_t env, float px, float py, double vx, double vy,
                                              bool vel_is_f32, double heading, double speed, double gx, double gy) {
  using R = real_t<FAITH>;
  const gca_config& c = a.cfg;
  if (c.obs_kind == GCA_OBS_NONE || c.obs_kind == GCA_OBS_NEAREST) return;
  const bool of = own_first(c);
  R* row = reinterpret_cast<R*>(a.obs) + env * (size_t)a.D;
  R* o = row + (of ? 0 : (c.obs_kind == GCA_OBS_RAW6 ? 6 : 4) * (size_t)a.s.N);
  // the eight entries of a goal-last row start on a 16-byte boundary (4 N or 6 N entries precede them in rows of
  // 4 N + 8 / 6 N + 8): they leave as 16-byte stores (two in f32, four in f64) instead of eight scalar ones
  auto store8 = [&](R v0, R v1, R v2, R v3, R v4, R v5, R v6, R v7) {
    if (reinterpret_cast<uintptr_t>(o) & 15u) {             // (6 N + 8 entries per row with N odd: every other row)
      o[0] = v0; o[1] = v1; o[2] = v2; o[3] = v3; o[4] = v4; o[5] = v5; o[6] = v6; o[7] = v7;
      return;
    }
    if constexpr (FAITH) {
      double2* q = reinterpret_cast<double2*>(o);
      q[0] = make_double2(v0, v1); q[1] = make_double2(v2, v3); q[2] = make_double2(v4, v5); q[3] = make_double2(v6, v7);
    } else {
      float4* q = reinterpret_cast<float4*>(o);
      q[0] = make_float4(v0, v1, v2, v3); q[1] = make_float4(v4, v5, v6, v7);
    }
  };
  if (c.obs_kind == GCA_OBS_RAW || c.obs_kind == GCA_OBS_RAW6) {
    store8((R)px, (R)py, (R)vx, (R)vy, (R)speed, (R)heading, (R)gx, (R)gy);
    return;
  }
  const Derived& k = a.k;
  const float nx = div_prepared(k, px, k.ob_w, k.inv_ob_w), ny = div_prepared(k, py, k.ob_h, k.inv_ob_h);
  R e2, e3;
  if (vel_is_f32) {
    e2 = (R)norm_vel_f32(k, (float)vx);
    e3 = (R)norm_vel_f32(k, (float)vy);
  } else {
    e2 = (R)norm_vel_f64(c, k, vx);
    e3 = (R)norm_vel_f64(c, k, vy);
  }
  const R e4 = (R)ddiv_prepared(k, __dadd_rn(speed, -c.ob_min_speed), k.dv_speed, k.rc_speed);
  const R e5 = (R)ddiv_prepared(k, heading, k.dv_2pi, k.rc_2pi);
  if (!of) {
    store8((R)nx, (R)ny, e2, e3, e4, e5, (R)ddiv_prepared(k, gx, k.dv_w, k.rc_w), (R)ddiv_prepared(k, gy, k.dv_h, k.rc_h));
    return;
  }
  o[0] = (R)nx;
  o[1] = (R)ny;
  o[2] = e2;
  o[3] = e3;
  o[4] = e4;
  o[5] = e5;
  R* ag = reinterpret_cast<R*>(a.achieved) + 2 * env;
  R* dg = reinterpret_cast<R*>(a.desired) + 2 * env;
  if (c.obs_kind == GCA_OBS_HER) {
    ag[0] = (R)nx; ag[1] = (R)ny;
    dg[0] = (R)ddiv_prepared(k, gx, k.dv_w, k.rc_w);
    dg[1] = (R)ddiv_prepared(k, gy, k.dv_h, k.rc_h);
  } else {
    ag[0] = (R)px; ag[1] = (R)py;
    dg[0] = (R)gx; dg[1] = (R)gy;
  }
}

// _get_ob() of Simulators/SingleAircraftDiscrete9HEREnv.py:106-165 for one env: ownship (x, y, vx, vy), then the
// Config.n nearest intruders, nearest first (ties: lowest index), each (x, y, vx, vy, dist / Config.diagonal), and the
// normalised achieved / desired goals.  Distances in the dtype the reference computes them in (f32 positions: f32
// norm; a retried spawn's f64 position: f64 norm), compared by value like np.argpartition / argsort of the mixed array.
// Four lanes per env: sub-lane q scans every 4th position unit into a private sorted list of the KN best, the four
// lists are merged by shuffles (every sub-lane ends with the same full list) and each sub-lane writes the entries of
// one winner - 4x the threads of a lane-per-env pass and 4x shorter chains.  The list is a branch-free insertion
// network on keys ordered by (distance, index): FAST packs the f32 distance bits (non-negative floats order like
// unsigned integers) and the index into one 64-bit word; FAITHFUL compares f32 / f64 distances by value as doubles.
// A list of the KN >= nearest_n best has the nearest_n best as its prefix.  Must be called by all 32 lanes of a warp;
// `valid` masks the envs past the end of the batch.
struct NearKeyF64 {
  double d;
  int i;
};
__device__ __forceinline__ bool near_less(const NearKeyF64& x, const NearKeyF64& y) {
  return x.d < y.d || (x.d == y.d && x.i < y.i);
}
__device__ __forceinline__ bool near_less(unsigned long long x, unsigned long long y) { return x < y; }
__device__ __forceinline__ NearKeyF64 near_shfl(const NearKeyF64& v, int src) {
  NearKeyF64 r;
  r.d = __shfl_sync(FULL, v.d, src);
  r.i = __shfl_sync(FULL, v.i, src);
  return r;
}
__device__ __forceinline__ unsigned long long near_shfl(unsigned long long v, int src) { return __shfl_sync(FULL, v, src); }

template <bool FAITH, int KN>
__device__ __forceinline__ void write_obs_nearest(const StepArgs& a, size_t env, const int q, const bool valid) {
  using R = real_t<FAITH>;
  using Key = typename std::conditional<FAITH, NearKeyF64, unsigned long long>::type;
  const DevState& s = a.s;
  const gca_config& c = a.cfg;
  const Derived& k = a.k;
  const int kn = c.nearest_n;
  const int plane = s.counters[env].z & 1;
  const float2 own = s.own_pos[env];
  Key slot[KN];
#pragma unroll
  for (int j = 0; j < KN; ++j) {
    if constexpr (FAITH) { slot[j].d = CUDART_INF; slot[j].i = INT_MAX; }
    else slot[j] = ~0ull;
  }
  auto consider = [&](Key key) {                          // sorted insertion: KN compare-exchanges, no branches
#pragma unroll
    for (int j = 0; j < KN; ++j) {
      const bool lt = near_less(key, slot[j]);
      const Key lo = lt ? key : slot[j], hi = lt ? slot[j] : key;
      slot[j] = lo;
      key = hi;
    }
  };
  // ---- scan: positions only (velocities are fetched for the winners)
  const uint8_t* pbase = s.ipos + (size_t)plane * s.pos_plane;
  if constexpr (FAITH) {
    for (int i = q; i < s.N; i += 4) {
      const double2 p = *reinterpret_cast<const double2*>(pbase + ipos_offset(s, true, env, i));
      const bool wide = (s.dflag[flag_index(s, env, i >> 5)] >> (i & 31)) & 1u;
      NearKeyF64 key;
      key.d = wide ? dist_f64((double)own.x, (double)own.y, p.x, p.y)
                   : (double)__fsqrt_rn(dist2_f32(own.x, own.y, (float)p.x, (float)p.y));
      key.i = i;
      consider(key);
    }
  } else {
    for (int i = 2 * q; i < s.N; i += 8) {                // a 16-byte unit holds intruders i and i + 1
      const float4 p = *reinterpret_cast<const float4*>(pbase + ipos_offset(s, false, env, i));
      const float d0 = __fsqrt_rn(dist2_f32(own.x, own.y, p.x, p.y)), d1 = __fsqrt_rn(dist2_f32(own.x, own.y, p.z, p.w));
      consider(((unsigned long long)__float_as_uint(d0) << 32) | (unsigned)i);
      if (i + 1 < s.N) consider(((unsigned long long)__float_as_uint(d1) << 32) | (unsigned)(i + 1));
    }
  }
  // ---- merge: every sub-lane inserts the ORIGINAL lists of the other three
  const int lane = threadIdx.x & 31, base = lane & ~3;
  Key orig[KN];
#pragma unroll
  for (int j = 0; j < KN; ++j) orig[j] = slot[j];
#pragma unroll
  for (int r = 1; r < 4; ++r) {
    const int src = base + ((q + r) & 3);
#pragma unroll
    for (int j = 0; j < KN; ++j) consider(near_shfl(orig[j], src));
  }
  // ---- output: sub-lane q writes winners q and q + 4; sub-lane 0 also the ownship entries, sub-lane 1 the goals
  R* row = reinterpret_cast<R*>(a.obs) + env * (size_t)a.D;
  const float nx = div_prepared(k, own.x, k.ob_w, k.inv_ob_w), ny = div_prepared(k, own.y, k.ob_h, k.inv_ob_h);
#pragma unroll
  for (int j = 0; j < KN; ++j) {
    if (valid && j < kn && (j & 3) == q) {
      int wi;
      double wd;
      if constexpr (FAITH) { wi = slot[j].i; wd = slot[j].d; }
      else { wi = (int)(unsigned)slot[j]; wd = (double)__uint_as_float((unsigned)(slot[j] >> 32)); }
      if (wi >= 0 && wi < s.N) {
        Intr<FAITH> it;
        load_intruder<FAITH>(s, plane, env, wi, it);
        bool wide = false;
        if constexpr (FAITH) wide = it.is64;
        R* o = row + 4 + 5 * j;
        if (wide) {
          o[0] = (R)ddiv_prepared(k, (double)it.px, k.dv_w, k.rc_w);
          o[1] = (R)ddiv_prepared(k, (double)it.py, k.dv_h, k.rc_h);
          o[4] = (R)__ddiv_rn(wd, c.ob_diagonal);
        } else {
          o[0] = (R)div_prepared(k, (float)it.px, k.ob_w, k.inv_ob_w);
          o[1] = (R)div_prepared(k, (float)it.py, k.ob_h, k.inv_ob_h);
          o[4] = (R)__fdiv_rn((float)wd, (float)c.ob_diagonal);
        }
        o[2] = (R)norm_vel_f32(k, it.vx);
        o[3] = (R)norm_vel_f32(k, it.vy);
      }
    }
  }
  if (valid && q == 0) {
    const double2 vel = s.own_vel[env];
    row[0] = (R)nx;
    row[1] = (R)ny;
    if (s.own_vel_f32[env]) {
      row[2] = (R)norm_vel_f32(k, (float)vel.x);
      row[3] = (R)norm_vel_f32(k, (float)vel.y);
    } else {
      row[2] = (R)norm_vel_f64(c, k, vel.x);
      row[3] = (R)norm_vel_f64(c, k, vel.y);
    }
  }
  if (valid && q == 1) {
    const double2 goal = s.goal[env];
    R* ag = reinterpret_cast<R*>(a.achieved) + 2 * env;
    R* dg = reinterpret_cast<R*>(a.desired) + 2 * env;
    ag[0] = (R)nx; ag[1] = (R)ny;
    dg[0] = (R)ddiv_prepared(k, goal.x, k.dv_w, k.rc_w);
    dg[1] = (R)ddiv_prepared(k, goal.y, k.dv_h, k.rc_h);
  }
}

// The f32 bit pattern of the relabel reward: -(d > goal_radius).astype(np.float32) (PKG/SingleAircraftHEREnv.py:194-196),
// -1.0 or -0.0, and (d < goal_radius).astype(np.float32) (PKG/SingleAircraftDiscreteHEREnv.py:184-186).  Selected and
// stored as integers: ptxas (CUDA 12.9, sm_100a) turned `selp.f32 -0.0, -1.0` of the f32 kernels into an integer
// select of 0 / -1 and an int-to-float conversion, which stores +0.0 where the reference returns -0.0.
__device__ __forceinline__ uint32_t relabel_reward_bits(int kind, bool gt, bool lt) {
  if (kind == GCA_OBS_HER) return gt ? 0xbf800000u : 0x80000000u;
  return lt ? 0x3f800000u : 0u;
}

}  // namespace gca
