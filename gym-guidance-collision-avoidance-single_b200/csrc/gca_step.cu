// gca_step.cu - step / reset / observe of the batched simulator (sm_100a).
//
// One step of a PHILOX handle = two launches on the caller's stream (tape replays: three, the ownship role as a kernel
// of its own; no intruders: one, step_n0_kernel), each part shaped for what bounds it:
//
//   ownship role           thread = env; the leading blocks of step_intruders_kernel's grid (tape handles:
//                          step_own_kernel).  Ownship kinematics (PKG/SingleAircraftEnv.py:299-309): all of it f64
//                          (Philox + Box-Muller, sincos, clamp).  Publishes the 16-byte record the streaming role
//                          waits for, then settles what the ownship alone decides (reward candidate, observation
//                          tail) while the stream is already running.  FP64 latency bound.
//   step_intruders_kernel  warp = 8 intruders x 32 envs, lane = env.  THE streaming pass: advance, map
//                          test, separation test on the squared distance, observation entries.  It
//                          reads one position plane and writes the other (gca_device.cuh), so it is
//                          order-free: work items are tiny (4 KB in, 6 KB out), there are ~10x more of
//                          them than resident warps, and the hardware block scheduler hands them to
//                          whichever SM drains fastest - which is what it takes to reach the DRAM
//                          roofline on a part whose GPCs do not get equal shares of the memory system
//                          (measured: with one resident warp per 32 envs the same arithmetic ended
//                          between 32 and 55 us depending on the SM).  Loads are 16 bytes per lane,
//                          512 contiguous bytes per warp instruction, 8 independent ones in flight per
//                          lane; positions leave the same way; observation entries are transposed
//                          through shared memory so that every store covers whole 32-byte sectors of
//                          the 1312-byte observation rows.  Events (an intruder left the map / is inside
//                          the separation or NMAC radius) are rare and only RECORDED here as bit masks.
//   step_finish_kernel     warp = 32 envs, lane = env.  Replays the reference's sequential loop
//                          semantics from the recorded masks (PKG/SingleAircraftEnv.py:149-170): first
//                          NMAC index wins and everything after it is put back where it was (Q9),
//                          a replaced intruder is tested with its old distance and starts with conflict False (Q7),
//                          the flag never clears otherwise (Q8); then the step's return (an intruder event outranks
//                          what the ownship role settled), counters, the scalar part of the VecEnv auto-reset; and
//                          in the same launch the spawn phase: one lane per respawn, one warp per 32 spawns of a
//                          reset (tape handles respawn in place, in the reference's draw order).
// Every byte of intruder state is read once and written once per step; nothing is staged in HBM except
// 16 bytes per env (ownship position for the streaming pass) and the event words.
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <utility>

#include "gca_device.cuh"
#include "gca_launch.h"
#include "gca_step_common.cuh"

namespace gca {

// Optional kernel-level timestamps (build with -DGCA_PHASE_TIMING): first block in / last block out per kernel.
#ifdef GCA_PHASE_TIMING
__device__ unsigned long long g_kstamp[8];   // [kernel][start, end] x 3, then the streaming pass's first record wait: begun, record seen
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ unsigned long long g_cta[8192 * 2];   // per block of the streaming kernel: first instruction, last instruction
extern "C" int gca_debug_cta(unsigned long long* host) { return (int)cudaMemcpyFromSymbol(host, g_cta, sizeof(g_cta)); }
// per tile: finish start, end, respawn records, resets, phase stamps.  Respawn records (PHILOX only; TAPE tiles leave the
// slot alone): the records the spawn phase ran, capped at kTileRespawnCap, including records of envs that reset and were
// skipped, excluding the respawns made in place (list full, or N > 128)
__device__ unsigned long long g_fin[2048 * 8];
extern "C" int gca_debug_fin(unsigned long long* host) { return (int)cudaMemcpyFromSymbol(host, g_fin, sizeof(g_fin)); }
__device__ unsigned int g_lat[8 * 64];            // position-load latency of the streaming pass: [eighth of the walk][64-cycle bucket]
extern "C" int gca_debug_lat(unsigned int* host, int clear) {
  int rc = (int)cudaMemcpyFromSymbol(host, g_lat, sizeof(g_lat));
  if (clear) { static unsigned int zero[8 * 64]; rc |= (int)cudaMemcpyToSymbol(g_lat, zero, sizeof(zero)); }
  return rc;
}
#define GCA_KSTAMP_IN(kid) do { if (threadIdx.x == 0) atomicMin(&g_kstamp[2 * (kid)], gtime()); } while (0)
#define GCA_KSTAMP_OUT(kid) do { if (threadIdx.x == 0) atomicMax(&g_kstamp[2 * (kid) + 1], gtime()); } while (0)
extern "C" int gca_debug_kstamps(unsigned long long* host, int reset) {
  int rc = (int)cudaMemcpyFromSymbol(host, g_kstamp, sizeof(g_kstamp));
  if (reset) {
    unsigned long long init[8] = {~0ull, 0, ~0ull, 0, ~0ull, 0, ~0ull, ~0ull};
    rc |= (int)cudaMemcpyToSymbol(g_kstamp, init, sizeof(init));
  }
  return rc;
}
#else
#define GCA_KSTAMP_IN(kid) do { } while (0)
#define GCA_KSTAMP_OUT(kid) do { } while (0)
#endif

constexpr int kChunkUnits = 4;                   // 16-byte units (intruder pairs) per lane and work item
constexpr int kChunkIntr = 2 * kChunkUnits;       // 8 intruders
constexpr int kTileRespawnCap = 128;              // respawn records per tile (32 envs) and step; beyond that the lane spawns in place
constexpr int kWarpsB = 4;                        // work items per block of the streaming pass
constexpr int kFaithMinBlocks = 1;                // blocks per SM the FAITHFUL streaming kernel is compiled for
// staging row of one lane: 8 intruders x 16 bytes of observation entries (FAITHFUL: 32 bytes), plus 16 bytes so that
// the row stride is an odd multiple of 16 (conflict-free 16-byte shared accesses across a quarter warp)
constexpr uint32_t kObsRow = 16u * kChunkIntr + 16u;
constexpr uint32_t kObsRow64 = 32u * kChunkIntr + 16u;
static_assert(32 % kChunkIntr == 0, "the event bits of a work item must not straddle a word, and the FAST write-out "
                                    "stores 32 / kChunkIntr whole env rows per instruction");
static_assert(32 * kChunkIntr == 16 * 16, "the FAITHFUL write-out stores one env's work item with 16 lanes x 16 bytes");
static_assert(kWarpsB * 32 * kObsRow64 <= 0xc000, "the FAITHFUL staging buffer must fit in static shared memory");

// spawn() of intruder i of env `env` (slot: i for reset_intruder() :229-238, GCA_SLOT_RESET | i for reset() :80-88) and
// its stores: position into `plane`, velocity, observation entries into the env's row `obase` (obs_intruder_base).
// Returns whether the position is f64 (Q3).
template <bool FAITH, bool TAPE>
__device__ __forceinline__ bool spawn_store(const StepArgs& a, Draws<TAPE>& d, uint32_t slot, size_t env, int i, int plane,
                                            float ox, float oy, real_t<FAITH>* obase) {
  const DevState& s = a.s;
  Intr<FAITH> it;
  spawn<FAITH, TAPE>(d, a.cfg, a.k, slot, ox, oy, it, ihs_slot(s, env, i));
  store_ipos<FAITH>(s, plane, env, i, it);
  store_ivel(s, env, i, it.vx, it.vy);
  write_obs_intruder<FAITH>(a, obase, i, it);
  return it.is64;
}

// reset()'s spawns of intruders 32 r .. 32 r + 31 of env `env`, one per lane, then the word's flags: conflict False,
// FAITHFUL the f64 bits of the new positions.  Executed by the whole warp; PHILOX only (the draws are independent).
template <bool FAITH>
__device__ __forceinline__ void spawn_reset_word(const StepArgs& a, Draws<false>& d, size_t env, int r, int lane, int plane,
                                                 const float2& own) {
  const DevState& s = a.s;
  const int i = r * 32 + lane;
  bool wide = false;
  if (i < s.N)
    wide = spawn_store<FAITH, false>(a, d, GCA_SLOT_RESET | (uint32_t)i, env, i, plane, own.x, own.y, obs_intruder_base<FAITH>(a, env));
  const uint32_t dw = __ballot_sync(FULL, wide);
  if (lane == 0) {
    s.cflag[flag_index(s, env, r)] = 0u;
    if constexpr (FAITH) s.dflag[flag_index(s, env, r)] = dw;
  }
}

// reset(): PKG/SingleAircraftEnv.py:66-98 for env `env`, executed by the whole warp; positions go to `plane`.
// PHILOX: lanes = intruders.  TAPE: lane `owner` replays the reference's sequential draw order.
template <bool FAITH, bool TAPE>
__device__ __forceinline__ void reset_env_warp(const StepArgs& a, size_t env, int plane, int lane, int owner,
                                               Draws<TAPE>& d, double2& goal, const float ox, const float oy) {
  const DevState& s = a.s;
  const gca_config& c = a.cfg;
  // (ox, oy): the ownship the new intruders keep their distance from - (50, 50) :72-76, or the random start
  if constexpr (TAPE) {
    if (lane == owner) {
      for (int r = 0; r < s.W; ++r) {
        uint32_t dw = 0;
        for (int j = 0; j < 32 && r * 32 + j < s.N; ++j) {
          const int i = r * 32 + j;
          const bool is64 = spawn_store<FAITH, TAPE>(a, d, GCA_SLOT_RESET | (uint32_t)i, env, i, plane, ox, oy, obs_intruder_base<FAITH>(a, env));
          dw |= (is64 ? 1u : 0u) << j;
        }
        s.cflag[flag_index(s, env, r)] = 0u;
        if constexpr (FAITH) s.dflag[flag_index(s, env, r)] = dw;
      }
      draw_goal(d, c, goal.x, goal.y);   // Goal(random_pos()) :93
    }
  } else {
    const float2 own = make_float2(ox, oy);
    for (int r = 0; r < s.W; ++r) spawn_reset_word<FAITH>(a, d, env, r, lane, plane, own);
    if (lane == owner) draw_goal(d, c, goal.x, goal.y);
  }
}

// reset() of every env of the warp's tile whose lane has `resets` set, one env at a time (the tape is sequential): the
// ownship's draws first, then the intruders' and the goal's (reset_env_warp), then lane e's draws continue behind them.
// On return a resetting lane holds its env's new pos / hs / vel / goal.  `nxt`: the plane the env's positions go to.
template <bool FAITH, bool TAPE>
__device__ __forceinline__ void reset_envs_warp(const StepArgs& a, size_t env0, int lane, bool resets, int nxt, Draws<TAPE>& d,
                                                float2& pos, double2& hs, double2& vel, double2& goal) {
  uint32_t rmask = __ballot_sync(FULL, resets);
  while (rmask) {
    const int e = __ffs(rmask) - 1;
    rmask &= rmask - 1;
    __syncwarp();                                                 // lane e's stores above come first
    Draws<TAPE> de = d;
    if constexpr (!TAPE) {
      de.env = __shfl_sync(FULL, d.env, e);
      de.tick = __shfl_sync(FULL, d.tick, e);
    }
    const int plane = __shfl_sync(FULL, nxt, e);
    if (lane == e) reset_ownship<TAPE>(a.cfg, de, pos, hs, vel);  // (its draws come first on the tape)
    const float rx = __shfl_sync(FULL, pos.x, e), ry = __shfl_sync(FULL, pos.y, e);
    reset_env_warp<FAITH, TAPE>(a, env0 + e, plane, lane, e, de, goal, rx, ry);
    if constexpr (TAPE) {
      if (lane == e) d = de;
    }
  }
}

// the ownship side of reset() for env `me`: its state, no_conflict and ep_steps zeroed, the reset observation's
// ownship / goal entries (f32 velocity, :76)
template <bool FAITH>
__device__ __forceinline__ void store_own_reset(const StepArgs& a, size_t me, float2 pos, double2 hs, double2 vel, double2 goal,
                                                int4& cnt) {
  const DevState& s = a.s;
  s.own_pos[me] = pos;
  s.own_hs[me] = hs;
  s.own_vel[me] = vel;
  s.own_vel_f32[me] = 1;
  s.goal[me] = goal;
  cnt.x = 0;
  cnt.y = 0;
  write_obs_own<FAITH>(a, me, pos.x, pos.y, vel.x, vel.y, true, hs.x, hs.y, goal.x, goal.y);
}

// ------------------------------------------------------------------------------ 1. ownship
// Ownship.step(a)   PKG/SingleAircraftEnv.py:299-309 (2Env :291-301, DiscreteHER :301-311) for env `me`.
// TAPE handles (parity replays): a kernel of its own, which also clears the env's event words.
// PHILOX handles: the ownship ROLE of step_intruders_kernel (the first blocks of its grid).  It publishes the 16-byte
// record the streaming role waits for - (x, y) first, then (bits, stamp) behind a fence - as soon as the new position
// is known, and then settles everything of the step that does not depend on the intruders while the streaming role is
// already running: the ownship / goal tail of the observation (:115-124) and the reward the step returns unless an
// intruder event outranks it (wall / goal / default / max steps, :173-183) -> DevState::pre.
template <bool FAITH, bool TAPE>
__device__ __forceinline__ void own_update(const StepArgs& a, const size_t me, const uint32_t stamp, const bool publish) {
  using R = real_t<FAITH>;
  const DevState& s = a.s;
  const gca_config& c = a.cfg;
  const Derived& k = a.k;
  float2 pos = s.own_pos[me];
  double2 hs = s.own_hs[me];
  int4 cnt = s.counters[me];
  double2 goal = make_double2(0., 0.);
  if constexpr (!TAPE) goal = s.goal[me];
  Draws<TAPE> d = make_draws<TAPE>(a, me, (uint32_t)cnt.z);
  double f0, f1 = 0.0;
  if (c.action_kind == GCA_ACT_CONTINUOUS2) {
    const R* act = reinterpret_cast<const R*>(a.actions) + 2 * me;
    f0 = (double)act[0];
    f1 = (double)act[1];
  } else {
    const int act = reinterpret_cast<const int*>(a.actions)[me];
    if (c.action_kind == GCA_ACT_DISCRETE9) {
      f0 = (double)(act / 3 - 1);
      f1 = (double)(act % 3 - 1);
    } else {
      f0 = (double)(act - 1);
    }
  }
  double nh, ns, sn, cs;
  draw_own_noise(d, c, nh, ns);
  double heading = __dadd_rn(hs.x, __dmul_rn(c.d_heading, f0));
  heading = __dadd_rn(heading, nh);
  double speed = c.action_kind == GCA_ACT_DISCRETE3 ? __dadd_rn(hs.y, c.speed_sigma)      // reference quirk Q16
                                                    : __dadd_rn(hs.y, __dmul_rn(c.d_speed, f1));
  const double m = c.max_speed < speed ? c.max_speed : speed;     // min(speed, max_speed)
  speed = m > c.min_speed ? m : c.min_speed;                      // max(min_speed, .)
  speed = __dadd_rn(speed, ns);                                   // noise after the clamp (Q5)
  gca_sincos(heading, &sn, &cs);
  const double2 vel = make_double2(__dmul_rn(speed, cs), __dmul_rn(speed, sn));
  hs = make_double2(heading, speed);
  pos = make_float2((float)__dadd_rn((double)pos.x, vel.x), (float)__dadd_rn((double)pos.y, vel.y));
  cnt.y += 1;                                                     // StackEnv :118
  const bool maxstep_hit = c.max_steps > 0 && cnt.y >= c.max_steps;   // StackEnv :134-136: the intruder loop never runs
  const uint32_t bits = (maxstep_hit ? 0u : kOwnRuns) | ((uint32_t)(cnt.z & 1) * kOwnPlane);
  if constexpr (TAPE) {
    s.own_b[me] = make_float4(pos.x, pos.y, __uint_as_float(bits), 0.f);
  } else if (publish) {
    // one 16-byte store, read with one 16-byte load: both are single transactions on one 32-byte sector, so a matching
    // stamp comes with its position (no fence: nothing else has to be visible to the streaming lanes)
    st_release_quad(reinterpret_cast<float*>(&s.own_b[me]), pos.x, pos.y, __uint_as_float(bits), __uint_as_float(stamp));
  }
  if constexpr (!TAPE) {                                         // (what the finish kernel loads first: kept in the L2)
    const uint64_t keep = l2_evict_last_policy();
    stg_stream2(&s.own_pos[me], pos.x, pos.y, keep);
    stg_stream(&s.counters[me], make_float4(__int_as_float(cnt.x), __int_as_float(cnt.y), __int_as_float(cnt.z), __int_as_float(cnt.w)), keep);
  } else {
    s.own_pos[me] = pos;
    s.counters[me] = cnt;
  }
  s.own_hs[me] = hs;
  s.own_vel[me] = vel;
  s.own_vel_f32[me] = 0;
  if constexpr (TAPE) {
    a.cursor[me] = d.cur;
    for (int w = 0; w < s.W; ++w) {
      const size_t fi = flag_index(s, me, w);
      s.ev_conf[fi] = 0u;
      s.ev_gone[fi] = 0u;
    }
    s.ev_nmac[me] = INT_MAX;
    if (c.shaped_nearest) s.ev_near[me] = 0x7f800000u;            // +inf
  } else {
    const Settled own = settle_own(c, k, maxstep_hit, pos, goal);
    const double pre_bits = __longlong_as_double((long long)(own.info | (own.done << 8)));
    stg_stream(&s.pre[me], make_float4(__int_as_float(__double2loint(own.reward)), __int_as_float(__double2hiint(own.reward)),
                                       __int_as_float(__double2loint(pre_bits)), __int_as_float(__double2hiint(pre_bits))),
               l2_evict_last_policy());
    write_obs_own<FAITH>(a, me, pos.x, pos.y, vel.x, vel.y, false, hs.x, hs.y, goal.x, goal.y);   // :115-124
  }
}

template <bool FAITH, bool TAPE>
__global__ void __launch_bounds__(128) step_own_kernel(const StepArgs a) {
  const DevState& s = a.s;
  pdl_wait();
  GCA_KSTAMP_IN(0);
  const size_t me = (size_t)blockIdx.x * 128 + threadIdx.x;
  if (me >= (size_t)s.T * 32) return;
  if (me >= (size_t)s.B) {                                // padding lanes of the last tile
    s.own_b[me] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  own_update<FAITH, TAPE>(a, me, 0u, false);
  GCA_KSTAMP_OUT(0);
}

// ------------------------------------------------------------------------------ finish (one warp, one tile)
// Replays the reference's sequential loop semantics for the 32 envs of `tile` from the event words that the
// streaming pass recorded, then rewards, observation tail, counters, auto-reset.  Called by the warp that
// completed the tile's last work item (or by step_finish_kernel when there are no intruders).  The event
// words were produced by other warps of the same launch: they are read with ld.global.cg (L2).
// per warp of step_finish_kernel (PHILOX): what the spawn phase of the same kernel needs of the tile's envs
struct WarpScratch {
  uint32_t list[kTileRespawnCap];   // (lane of the env << 8 | intruder): the intruders that left the map in this step
  float2 pos[32];                   // the ownship the respawns keep their distance from (this step's position)
  int tick[32];                     // tick of this step; -1: the env finished and was reset (its respawns are moot)
  int n_jobs;
};
struct BlockScratch {               // per block: the envs that finished under auto-reset (their N spawns, one warp per 32)
  int env[128];
  int tick[128];                    // the tick of the step that finished the env
  float2 pos[128];                  // the ownship its new intruders keep their distance from (reset position)
  int count;
};

template <bool FAITH, bool TAPE>
__device__ __forceinline__ void finish_tile(const StepArgs& a, const int tile, const int lane, WarpScratch* ws,
                                            BlockScratch* bs) {
  using R = real_t<FAITH>;
  constexpr bool PRE = !TAPE;                             // the ownship role already settled the intruder-free part
  const DevState& s = a.s;
  const gca_config& c = a.cfg;
  const Derived& k = a.k;
  const size_t env0 = (size_t)tile * 32;
  const bool has_env = env0 + lane < (size_t)s.B;
  const size_t me = has_env ? env0 + lane : env0;
#ifdef GCA_PHASE_TIMING
  const unsigned long long fin_t0 = gtime();
  int fin_resets = 0;
#endif

  float2 pos = make_float2(0.f, 0.f);
  double2 hs = make_double2(0., 0.), vel = make_double2(0., 0.), goal = make_double2(0., 0.), pre = make_double2(0., 0.);
  int4 cnt = make_int4(0, 0, 0, 0);
  int stop = INT_MAX;
  uint32_t near_bits = 0x7f800000u;                       // FAST + shaped_nearest: smallest squared distance of the step (+inf: none)
  constexpr int kWordsAhead = 4;                          // N <= 128: the env's event / flag words live in registers
  uint32_t wc[kWordsAhead], wg[kWordsAhead], wf[kWordsAhead];
#pragma unroll
  for (int w = 0; w < kWordsAhead; ++w) wc[w] = wg[w] = wf[w] = 0u;
  if (has_env) {
    // everything this lane needs is requested before any of it is looked at: one round trip
    pos = s.own_pos[me];
    if constexpr (PRE) {
      pre = s.pre[me];
    } else {
      hs = s.own_hs[me];
      vel = s.own_vel[me];
      goal = s.goal[me];
    }
    cnt = s.counters[me];
    if (s.N > 0) {
      stop = __ldcg(&s.ev_nmac[me]);
#pragma unroll
      for (int w = 0; w < kWordsAhead; ++w) {
        if (w < s.W && s.W <= kWordsAhead) {              // (N > 128: the word-by-word path below reads and clears them)
          const size_t fi = flag_index(s, me, w);
          wc[w] = __ldcg(&s.ev_conf[fi]);
          wg[w] = __ldcg(&s.ev_gone[fi]);
          wf[w] = s.cflag[fi];
          if constexpr (PRE) {                            // consumed: the words are clear again for the next step
            if (wc[w]) s.ev_conf[fi] = 0u;
            if (wg[w]) s.ev_gone[fi] = 0u;
          }
        }
      }
      if constexpr (!FAITH) {
        if (c.shaped_nearest) near_bits = __ldcg(&s.ev_near[me]);
      }
      if constexpr (PRE) {
        if (stop != INT_MAX) s.ev_nmac[me] = INT_MAX;
        if (near_bits != 0x7f800000u) s.ev_near[me] = 0x7f800000u;
      }
    }
  }
  Draws<TAPE> d = make_draws<TAPE>(a, me, (uint32_t)cnt.z);
#ifdef GCA_PHASE_TIMING
  unsigned long long fin_t1 = 0, fin_t2 = 0, fin_t3 = 0;
  if (__any_sync(FULL, cnt.z + stop + (int)wc[0] + (int)wg[0] + (int)wf[0] + (int)goal.x == -12345)) fin_t1 = 1;   // consume the loads
  fin_t1 += gtime();
#endif
  const int cur = cnt.z & 1, nxt = cur ^ 1;               // nxt: the plane this step wrote = the env's next current plane
  const bool maxstep_hit = c.max_steps > 0 && cnt.y >= c.max_steps;
  const bool replay = has_env && !maxstep_hit && s.N > 0; // the reference's intruder loop ran for this env
  R* obase = obs_intruder_base<FAITH>(a, me);
  // the loop (PKG/SingleAircraftEnv.py:149-170) returned right after intruder `stop` (Q9): later events never happened
  const bool nmac = replay && stop != INT_MAX;
  bool conf_any = false;
  int newconf = 0;
  const bool words_in_regs = s.W <= kWordsAhead;
  const bool compact = !TAPE && words_in_regs && s.N > 0 && s.B <= (1 << 24);   // PHILOX draws do not depend on the visiting order

  auto visited_mask = [&](int w) -> uint32_t {
    const int lo = w * 32;
    return stop >= lo + 31 ? 0xffffffffu : (stop < lo ? 0u : (2u << (stop - lo)) - 1u);
  };
  // reset_intruder() for intruder i of this lane's env   :153-154, :229-238
  auto respawn_own = [&](int i, uint32_t& set64) {
    set64 |= (spawn_store<FAITH, TAPE>(a, d, (uint32_t)i, me, i, nxt, pos.x, pos.y, obase) ? 1u : 0u) << (i & 31);
  };
  // the loop's events in word w of this lane's env (conf, gone: the visited intruders; cf: the conflict word before the
  // step).  in_place: respawn here, in index order (TAPE: the reference's draw order); else the spawn phase does it.
  auto replay_word = [&](int w, uint32_t conf, uint32_t gone, uint32_t cf, bool in_place) {
    const size_t fi = flag_index(s, me, w);
    newconf += __popc(conf & ~cf);                        // False -> True transitions :161-163 (old object's flag, Q7)
    conf_any |= conf != 0u;
    const uint32_t ncf = (cf | conf) & ~gone;             // the flag never clears (Q8); a replaced intruder starts False
    if (ncf != cf) s.cflag[fi] = ncf;
    uint32_t set64 = 0;
    if (in_place) {
      uint32_t rest = gone;
      while (rest) {
        const int j = __ffs(rest) - 1;
        rest &= rest - 1;
        respawn_own(w * 32 + j, set64);
      }
    }
    if constexpr (FAITH) {
      if (gone) s.dflag[fi] = (s.dflag[fi] & ~gone) | set64;
    }
  };

  // self.dist_nearest_intruder (Simulators/SingleAircraftDiscrete3HEREnv.py:185,191): min over the intruders the loop
  // visited of the distance it measured - the advanced position of the OLD object, which the plane this step wrote
  // still holds for every intruder (respawns come later).  Python's min(d, current) keeps d on ties; value and dtype.
  double dnear = 9999.0;
  bool near64 = true, near_set = false;
  if (c.shaped_nearest && replay) {
    const uint8_t* pbase = s.ipos + (size_t)nxt * s.pos_plane;
    if constexpr (!FAITH) {
      // FAST: one dtype.  Without an NMAC every intruder was visited: sqrt of the smallest squared distance the
      // streaming pass recorded (sqrt is monotone).  After an NMAC at `stop` the visited prefix has no other distance
      // below NMAC_dist (it would have ended the loop earlier), so the minimum is the distance of `stop` itself.
      if (stop == INT_MAX) {
        dnear = (double)__fsqrt_rn(__uint_as_float(near_bits));
      } else {
        const float2 p = *reinterpret_cast<const float2*>(pbase + ipos_offset(s, false, me, stop));
        dnear = (double)__fsqrt_rn(dist2_f32(pos.x, pos.y, p.x, p.y));
      }
      near64 = false; near_set = true;
    } else {
      const int last = stop < s.N - 1 ? stop : s.N - 1;
      for (int i = 0; i <= last; ++i) {
        const double2 p = *reinterpret_cast<const double2*>(pbase + ipos_offset(s, true, me, i));
        const bool wide = (s.dflag[flag_index(s, me, i >> 5)] >> (i & 31)) & 1u;
        const double dd = wide ? dist_f64((double)pos.x, (double)pos.y, p.x, p.y)
                               : (double)__fsqrt_rn(dist2_f32(pos.x, pos.y, (float)p.x, (float)p.y));
        if (!(dnear < dd)) { dnear = dd; near64 = wide; near_set = true; }
      }
    }
  }
  if (replay) {
    if (words_in_regs) {
#pragma unroll
      for (int w = 0; w < kWordsAhead; ++w) {
        const uint32_t vis = visited_mask(w);
        const uint32_t conf = wc[w] & vis, gone = wg[w] & vis;
        wg[w] = gone;
        if (conf | gone) replay_word(w, conf, gone, wf[w], !compact);
      }
    } else {
      for (int w = 0; w < s.W; ++w) {                     // N > 128: word by word
        const uint32_t vis = visited_mask(w);
        const size_t fi = flag_index(s, me, w);
        const uint32_t conf_all = __ldcg(&s.ev_conf[fi]), gone_all = __ldcg(&s.ev_gone[fi]);
        if constexpr (PRE) {
          if (conf_all) s.ev_conf[fi] = 0u;
          if (gone_all) s.ev_gone[fi] = 0u;
        }
        const uint32_t conf = conf_all & vis, gone = gone_all & vis;
        if (conf | gone) replay_word(w, conf, gone, s.cflag[fi], true);
      }
    }
  }
  // PHILOX: a respawn depends on nothing but (env, tick, intruder) and the ownship position, so the spawns
  // (FP64-heavy, 0-3 per env) are not done here, one lane per env, but queued for spawn_kernel, which runs one
  // lane per spawn over the whole batch.  The records go to the tile's own segment of the respawn list.
  int job_mine = 0, job_off = 0, job_total = 0;
  if constexpr (!TAPE) {
    if (compact) {
      if (replay) job_mine = __popc(wg[0]) + __popc(wg[1]) + __popc(wg[2]) + __popc(wg[3]);
      job_off = job_mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, job_off, o);
        if (lane >= o) job_off += t;
      }
      job_total = __shfl_sync(FULL, job_off, 31);
      job_off -= job_mine;
      // the records go to the warp's shared scratch: the spawn phase of the same kernel runs them one lane each
    }
    if (lane == 0) ws->n_jobs = job_total < kTileRespawnCap ? job_total : kTileRespawnCap;   // (0 when the spawns were made in place)
  }
#ifdef GCA_PHASE_TIMING
  fin_t2 = gtime();
#endif
  bool done = false;
  if (has_env) {
    if (nmac && !a.auto_reset) {
      // intruders after `stop` were never touched by the reference: put them back where they were
      // (under auto-reset the env is finished and all of its intruders are about to be replaced)
      for (int i = stop + 1; i < s.N; ++i) {
        Intr<FAITH> old;
        load_intruder<FAITH>(s, cur, me, i, old);
        store_ipos<FAITH>(s, nxt, me, i, old);
        write_obs_intruder<FAITH>(a, obase, i, old);
      }
    }
    cnt.x += newconf;
    // _terminal_reward()   :143-184 and the variant rows of SURVEY.md 8(a)
    double reward;
    int info;
    bool is_default = false;                               // the `return -dist/1200, False, ''` row: the nearest-intruder term applies
    if (maxstep_hit) {
      reward = 0.0; done = true; info = GCA_INFO_MAXSTEPS;
    } else if (nmac) {
      reward = c.r_nmac; done = true; info = GCA_INFO_NMAC;
    } else if (conf_any) {
      reward = c.r_conflict; info = GCA_INFO_CONFLICT;
    } else if constexpr (PRE) {                            // wall / goal / default: settled by the ownship role (own_update)
      const int bits = (int)__double_as_longlong(pre.y);
      reward = pre.x; info = bits & 0xff; done = (bits >> 8) != 0;
      is_default = info == GCA_INFO_NONE;
    } else {
      const Settled own = settle_own(c, k, false, pos, goal);
      reward = own.reward; info = own.info; done = own.done != 0;
      is_default = info == GCA_INFO_NONE;
    }
    if (is_default && c.shaped_nearest) {                  // :225-232 (NumPy 2 weak scalars: an f32 distance stays f32)
      const double thr = 3 * c.minimum_separation;
      const bool lt = near_set ? (near64 ? dnear < thr : (float)dnear < (float)thr) : dnear < thr;
      if (lt) {
        if (near64) {
          const double r = __dadd_rn(__dmul_rn(c.conflict_coeff, dnear), -0.1);
          reward = __dadd_rn(reward, r);
        } else {
          const float r = __fadd_rn(__fmul_rn((float)c.conflict_coeff, (float)dnear), -(float)0.1);
          reward = c.shaped_default ? __dadd_rn(reward, (double)r) : (double)__fadd_rn((float)c.r_default, r);
        }
      }
    }
    if (c.time_limit > 0 && cnt.y >= c.time_limit) done = true;    // gym TimeLimit of the registered ids
    reinterpret_cast<R*>(a.reward)[me] = (R)reward;
    a.done[me] = done ? 1 : 0;
    a.info[me] = (uint8_t)info;
    if (a.nearest) reinterpret_cast<R*>(a.nearest)[me] = (R)dnear;
    if constexpr (!PRE) {                                          // (PRE: own_update wrote it; a reset overwrites it below)
      if (!(done && a.auto_reset))                                 // (a finished env shows its reset observation, below)
        write_obs_own<FAITH>(a, me, pos.x, pos.y, vel.x, vel.y, false, hs.x, hs.y, goal.x, goal.y);   // :115-124
    }
  }
  if constexpr (PRE) {                                             // for the spawn phase (before a reset replaces pos)
    ws->pos[lane] = pos;
    ws->tick[lane] = (has_env && !(done && a.auto_reset)) ? cnt.z : -1;
  }

  if constexpr (!TAPE) {
    if (compact && job_total > 0) {
      if (job_mine > 0) {
        uint32_t set64_own[kWordsAhead] = {0u, 0u, 0u, 0u};
        int at = job_off;
#pragma unroll
        for (int w = 0; w < kWordsAhead; ++w) {
          uint32_t rest = wg[w];
          while (rest) {
            const int j = __ffs(rest) - 1;
            rest &= rest - 1;
            if (at < kTileRespawnCap) ws->list[at] = ((uint32_t)lane << 8) | (uint32_t)(w * 32 + j);
            else if (!(done && a.auto_reset)) respawn_own(w * 32 + j, set64_own[w]);   // (list full: > 4 respawns per env on average)
            ++at;
          }
        }
        if constexpr (FAITH) {
#pragma unroll
          for (int w = 0; w < kWordsAhead; ++w)
            if (set64_own[w]) atomicOr(&s.dflag[flag_index(s, me, w)], set64_own[w]);
        }
      }
    }
  }
  if constexpr (TAPE) {
    // _update_headings() (Simulators/SingleAircraftMCTSRandIntruderEnv.py:166-174): step() runs it after
    // _terminal_reward whatever that returned, on the current intruder list, in index order - on the tape its draws
    // sit between the loop's respawns and the VecEnv reset's.  (PHILOX: turn_obs_kernel, one lane per intruder.)
    if (c.intruder_turns && has_env && s.ihs) {
      for (int i = 0; i < s.N; ++i) {
        const double p = d.next();
        if (!(p < c.turn_prob)) continue;
        const double raw = d.next();                                // np.random.uniform(-10, 10) as recorded
        double2 ih = s.ihs[ihs_index(s, me, i)];
        double sn, cs;
        ih.x = __dadd_rn(ih.x, __dmul_rn(raw, 3.141592653589793 / 180.0));   // math.radians
        gca_sincos(ih.x, &sn, &cs);
        s.ihs[ihs_index(s, me, i)] = ih;
        store_ivel(s, me, i, (float)__dmul_rn(ih.y, cs), (float)__dmul_rn(ih.y, sn));
      }
    }
  }
#ifdef GCA_PHASE_TIMING
  fin_t3 = gtime();
#endif
  // ---- VecEnv auto-reset: the observation handed back for a finished env is reset()'s (dummy_vec_env.py:52-55)
  const bool resets = a.auto_reset && has_env && done;
  int reset_slot = -1;
  if constexpr (TAPE) {
    reset_envs_warp<FAITH, TAPE>(a, env0, lane, resets, nxt, d, pos, hs, vel, goal);
  } else {
    // PHILOX: the 80 spawns of each finished env are independent of everything else; they are queued for
    // reset_spawn_kernel (one warp per 32 of them, all finished envs of the batch at once) instead of
    // serialising this warp.  The scalar part of reset() happens here.
    const uint32_t rmask = __ballot_sync(FULL, resets);
    if (rmask) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&bs->count, __popc(rmask));
      base = __shfl_sync(FULL, base, 0);
      if (resets) {
        reset_slot = base + __popc(rmask & ((1u << lane) - 1u));
        bs->env[reset_slot] = (int)me;
        draw_goal(d, c, goal.x, goal.y);   // Goal(random_pos()) :93
      }
#ifdef GCA_PHASE_TIMING
      fin_resets += __popc(rmask);
#endif
    }
  }
  if (resets) {
    if constexpr (!TAPE) {
      reset_ownship<TAPE>(c, d, pos, hs, vel);
      if (reset_slot >= 0) {                                          // (the spawn phase reads them from shared memory)
        bs->pos[reset_slot] = pos;
        bs->tick[reset_slot] = cnt.z;
      }
    }
    cnt.w += 1;
    store_own_reset<FAITH>(a, me, pos, hs, vel, goal, cnt);
  }
  if (has_env) {
    cnt.z += 1;                                                     // Philox tick; also flips the current position plane
    s.counters[me] = cnt;
    if constexpr (TAPE) a.cursor[me] = d.cur;
  }
#ifdef GCA_PHASE_TIMING
  if (lane == 0 && tile < 2048) {
    g_fin[tile * 8 + 0] = fin_t0; g_fin[tile * 8 + 1] = gtime(); g_fin[tile * 8 + 3] = fin_resets;
    g_fin[tile * 8 + 4] = fin_t1; g_fin[tile * 8 + 5] = fin_t2; g_fin[tile * 8 + 6] = fin_t3;
  }
#endif
}

// The spawn phase of a PHILOX step, run by the warps that just finished their tiles (no kernel of its own: a launch
// boundary costs more than this work).  (i) reset_intruder() (PKG/SingleAircraftEnv.py:153-154, :229-238) for every
// intruder of the tile that left the map, one LANE per spawn (records in the warp's scratch, ~14 per tile and step);
// (ii) after a block-wide barrier, reset()'s N spawns (:80-88) of every env of the block that finished under
// auto-reset, one WARP per 32 of them, whichever warp is free.  A spawn depends on (env, tick, intruder) and the
// ownship position only, so who executes it does not matter.
template <bool FAITH>
__device__ __forceinline__ void spawn_phase(const StepArgs& a, const int tile, const int wib, const int lane,
                                            WarpScratch* ws, BlockScratch* bs) {
  const DevState& s = a.s;
  Draws<false> d;
  d.k0 = a.key0; d.k1 = a.key1;
  if (tile < s.T) {
    __syncwarp();                                           // the records and per-env scratch of finish_tile
    const int n_resp = ws->n_jobs;
    for (int at = lane; at < n_resp; at += 32) {
      const uint32_t rec = ws->list[at];
      const int e = (int)(rec >> 8), i = (int)(rec & 0xffu);
      const int tick = ws->tick[e];
      if (tick < 0) continue;                               // the env finished and was reset: all its intruders are new anyway
      const size_t env = (size_t)tile * 32 + e;
      const float2 own = ws->pos[e];
      d.env = a.env_id0 + (uint32_t)env;
      d.tick = (uint32_t)tick;
      const bool is64 = spawn_store<FAITH, false>(a, d, (uint32_t)i, env, i, (tick & 1) ^ 1, own.x, own.y,   // (the plane this step wrote)
                                                  obs_intruder_base<FAITH>(a, env));
      if constexpr (FAITH) {
        if (is64) atomicOr(&s.dflag[flag_index(s, env, i >> 5)], 1u << (i & 31));
      }
    }
  }
#ifdef GCA_PHASE_TIMING
  if (lane == 0 && tile < 2048 && tile < s.T) {
    g_fin[tile * 8 + 2] = ws->n_jobs;
    g_fin[tile * 8 + 7] = gtime();
  }
#endif
  __syncthreads();                                          // every warp's resets are queued, their scalar state stored
  const int rounds = s.W, total = bs->count * rounds;
  for (int job = wib; job < total; job += 4) {
    const size_t env = (size_t)bs->env[job / rounds];
    const int r = job % rounds;
    const int tick = bs->tick[job / rounds];                // the tick of the step that finished the env
    d.env = a.env_id0 + (uint32_t)env;
    d.tick = (uint32_t)tick;
    spawn_reset_word<FAITH>(a, d, env, r, lane, (tick & 1) ^ 1, bs->pos[job / rounds]);   // (the plane this step wrote)
  }
}

// TAPE: finish only (respawns / resets replay the tape in place).  PHILOX: finish + spawn phase; the last kernel of
// the step's fixed part, so it also counts the step (DevState::step_seq, the stamp of the next step's ownship records).
template <bool FAITH, bool TAPE>
__global__ void __launch_bounds__(128) step_finish_kernel(const __grid_constant__ StepArgs a) {
  __shared__ WarpScratch ws[TAPE ? 1 : 4];
  __shared__ BlockScratch bs;
  if (!TAPE && threadIdx.x == 0) bs.count = 0;
  pdl_wait();
  GCA_KSTAMP_IN(2);
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tile = (long long)blockIdx.x * 4 + wib;
  if constexpr (TAPE) {
    if (tile < a.s.T) finish_tile<FAITH, TAPE>(a, (int)tile, lane, nullptr, nullptr);
  } else {
    __syncthreads();
    if (tile < a.s.T) finish_tile<FAITH, TAPE>(a, (int)tile, lane, &ws[wib], &bs);
    if (a.s.N > 0) spawn_phase<FAITH>(a, (int)(tile < a.s.T ? tile : a.s.T), wib, lane, &ws[wib], &bs);
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.s.step_seq += 1u;
  }
  GCA_KSTAMP_OUT(2);
}

// No intruders (the package default, PKG/config.py:8 `intruder_size = 0`), PHILOX: nothing runs between the ownship
// update and the finish, so the whole step is ONE kernel, thread = env (warp = tile, as in the finish).
// Two builds: MINB = 1 (94 registers, 5 blocks per SM: the shortest chain - batches that fit the GPU in a wave or two
// are bound by that latency: 5.3 us per step at 65,536 envs) and MINB = 8 (64 registers with a few spills, 8 blocks per
// SM: once the batch is many waves deep the kernel is bound by memory latency at low occupancy, and 32 instead of 20
// warps per SM take the 4 Mi-env step from 230 to 166 us = 61 % of the measured HBM peak on its 155 B per env-step).
template <bool FAITH, int MINB>
__global__ void __launch_bounds__(128, MINB) step_n0_kernel(const __grid_constant__ StepArgs a) {
  __shared__ WarpScratch ws[4];
  __shared__ BlockScratch bs;
  if (threadIdx.x == 0) bs.count = 0;
  pdl_wait();
  __syncthreads();
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tile = (long long)blockIdx.x * 4 + wib;
  const size_t me = (size_t)tile * 32 + lane;
  if (me < (size_t)a.s.B) own_update<FAITH, false>(a, me, 0u, false);
  if (tile < a.s.T) finish_tile<FAITH, false>(a, (int)tile, lane, &ws[wib], &bs);   // (reads back what this thread stored)
}

// ------------------------------------------------------------------------------ 2. intruders (the streaming pass)
// OM: 1 = the observation is GCA_OBS_VECTOR with the one-correction division exact (the registered ids'
// layout; FAST only): entries are computed without run-time layout tests and leave through the transposed
// shared-memory write-out.  2 = the same for the own-first layouts GCA_OBS_HER / GCA_OBS_DHER, whose intruder
// entries start 24 bytes into the row: 8-byte stores.  0 = generic (any layout, both modes): per-lane stores.
// DRIFT: every advance adds Config.position_sigma to the velocity (the random-intruder env); generic layout only, so the
// instruction streams of the other instantiations are what they were without it.
template <bool FAITH, int OM, bool DRIFT = false>
__global__ void __launch_bounds__(kWarpsB * 32, FAITH ? kFaithMinBlocks : 1) step_intruders_kernel(const __grid_constant__ StepArgs a) {
  static_assert(!(DRIFT && OM), "a handle with a position drift takes the generic observation path");
  pdl_wait();
  GCA_KSTAMP_IN(1);
#ifdef GCA_PHASE_TIMING
  if (threadIdx.x == 0 && blockIdx.x < 8192) g_cta[2 * blockIdx.x] = gtime();
#endif
  using R = real_t<FAITH>;
  static_assert(!(FAITH && OM), "the specialised observation path is FAST only");
  // observation staging: FAST specialised layouts 8 x 16 bytes per lane, FAITHFUL 8 x 32 bytes per lane (+ 16: odd stride)
  constexpr uint32_t kWarpSmem = OM ? 32 * kObsRow : (FAITH ? 32 * kObsRow64 : 16);
  constexpr uint32_t kStageBytes = kWarpsB * kWarpSmem;
  __shared__ __align__(16) uint8_t stage_smem[kStageBytes];
  const DevState& s = a.s;
  const Derived& k = a.k;
  // ---- PHILOX handles: the first own_blocks blocks of the grid are the OWNSHIP ROLE (thread = env).  Blocks are
  // dispatched in index order, so every record a streaming lane waits for below belongs to a block that is already
  // running or done (the forward-progress argument of a decoupled look-back scan).
  uint32_t stamp = 0u;
  if (a.own_blocks > 0) {
    stamp = *s.step_seq + 1u;
    if (blockIdx.x < (unsigned)a.own_blocks) {
      GCA_KSTAMP_IN(0);
      // (odd steps walk the batch backwards, like the streaming role below: the records needed first come first)
      const size_t env = (size_t)((stamp & 1u) ? (unsigned)a.own_blocks - 1u - blockIdx.x : blockIdx.x) * (kWarpsB * 32) + threadIdx.x;
      if (env < (size_t)s.B) {
        own_update<FAITH, false>(a, env, stamp, true);
      } else if (env < (size_t)s.T * 32) {                // padding lanes of the last tile
        st_release_quad(reinterpret_cast<float*>(&s.own_b[env]), 0.f, 0.f, 0.f, __uint_as_float(stamp));
      }
      GCA_KSTAMP_OUT(0);
      return;
    }
  }
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int n_chunks = (s.U + kChunkUnits - 1) / kChunkUnits;
  const long long work = (long long)(blockIdx.x - (unsigned)a.own_blocks) * kWarpsB + wib;
  do {                                                    // (one pass; `break` = this warp has no work item)
  if (work >= (long long)s.T * n_chunks) break;
  // Philox handles walk the tiles forwards in even steps and backwards in odd ones: the plane this step reads is the
  // plane the previous step wrote, and what it wrote LAST is what is most likely still in the L2 (43.3 -> 42.6 us)
  const int tile_fwd = (int)(work / n_chunks), ch = (int)(work - (long long)tile_fwd * n_chunks);
  const int tile = (a.own_blocks > 0 && (stamp & 1u)) ? s.T - 1 - tile_fwd : tile_fwd;
  const size_t me = (size_t)tile * 32 + lane;
  const bool has_env = me < (size_t)s.B;
  const int u0 = ch * kChunkUnits, i0 = 2 * u0;
  const int n_here = min(kChunkIntr, s.N - i0);           // intruders of this work item
  constexpr size_t kPosUnits = FAITH ? 2 : 1;
  const size_t unit0 = (size_t)tile * s.U + u0;           // first unit of this work item in the tile-planar order
  const uint8_t* vsrc = s.ivel + (unit0 * 32 + lane) * 16;
  // The velocity loads need nothing from the ownship record: they are issued first, so that they travel while the
  // record (which says which position plane is current) is still on its way.
  const uint64_t pol = l2_evict_first_policy();
  float4 vv[kChunkUnits];
  const bool full = !FAITH && n_here == kChunkIntr;
  if (full) {
#pragma unroll
    for (int g = 0; g < kChunkUnits; ++g) vv[g] = ldg_stream(vsrc + g * 512, pol);
  }
  float4 ob;
  GCA_KSTAMP_IN(3);                                       // (timing builds: first streaming block in / first record seen)
  if (a.own_blocks > 0) {
    // wait for this step's ownship record of the lane's env: it is stored with one 16-byte store and read with one
    // 16-byte aligned vector load, both served from one sector - a matching stamp comes with its position
    int spins = 0;
    for (;;) {
      ob = ld_volatile_f4(&s.own_b[me]);
      if (__all_sync(FULL, __float_as_uint(ob.w) == stamp)) break;
      if (++spins > (1 << 22)) {                          // ~0.5 s: dispatch order broke - fail loudly, do not hang
        if (lane == 0) atomicExch(s.error_flag, 1);
        break;
      }
      __nanosleep(32);
    }
  } else {
    ob = s.own_b[me];
  }
#ifdef GCA_PHASE_TIMING
  if (threadIdx.x == 0) { atomicMin(&g_kstamp[7], gtime()); }
#endif
  const uint32_t bits = __float_as_uint(ob.z);
  const bool runs = (bits & kOwnRuns) != 0;               // false: the reference's loop never ran for this env (max steps)
  const int par = (bits & kOwnPlane) ? 1 : 0;
  const float ox = ob.x, oy = ob.y;
  const size_t pos_off = (unit0 * kPosUnits * 32 + lane) * 16;
  const uint8_t* psrc = s.ipos + (size_t)par * s.pos_plane + pos_off;
  uint8_t* pdst = s.ipos + (size_t)(par ^ 1) * s.pos_plane + pos_off;
  R* obase = obs_intruder_base<FAITH>(a, me);
  uint32_t gone = 0, conf = 0, nmac = 0;                  // bit j: intruder i0 + j
  float near2 = __uint_as_float(0x7f800000u);             // FAST + shaped_nearest: smallest squared distance of this item

  bool fast_done = false;
  if constexpr (!FAITH) {
    if (full) {
      // ---- all 8 intruders at once, straight-line
      fast_done = true;
      float4 p[kChunkUnits], np[kChunkUnits];
#ifdef GCA_PHASE_TIMING
      const long long lat_t0 = clock64();
#endif
#pragma unroll
      for (int g = 0; g < kChunkUnits; ++g) p[g] = ldg_stream(psrc + g * 512, pol);
#ifdef GCA_PHASE_TIMING
      {
        float sink = 0.f;
        for (int g = 0; g < kChunkUnits; ++g) sink += p[g].x + p[g].w;
        if (__any_sync(FULL, sink == 1.2345e38f)) atomicAdd(&g_lat[0], 1u);   // (never true: makes the warp wait for the data here)
        const long long dt = clock64() - lat_t0;
        if (lane == 0) atomicAdd(&g_lat[min(7, tile_fwd * 8 / s.T) * 64 + (int)min(63ll, dt >> 6)], 1u);
      }
#endif
      const uint32_t wbits = __float_as_uint(k.win_w), hbits = __float_as_uint(k.win_h);
#pragma unroll
      for (int g = 0; g < kChunkUnits; ++g) {
        float4 dv = vv[g];
        if constexpr (DRIFT)                                // position += velocity + position_sigma (f32 sum first)
          dv = make_float4(__fadd_rn(dv.x, k.drift_f), __fadd_rn(dv.y, k.drift_f), __fadd_rn(dv.z, k.drift_f),
                           __fadd_rn(dv.w, k.drift_f));
        np[g] = make_float4(__fadd_rn(p[g].x, dv.x), __fadd_rn(p[g].y, dv.y),      // position += velocity :150
                            __fadd_rn(p[g].z, dv.z), __fadd_rn(p[g].w, dv.w));
        // 0 <= x <= W on f32 bit patterns (:153): a non-negative float is <= W iff its pattern is (as unsigned);
        // negatives and NaN have larger patterns (FAST positions are never -0.0, see gca_set_state).
        const bool oob0 = (__float_as_uint(np[g].x) > wbits) | (__float_as_uint(np[g].y) > hbits);
        const bool oob1 = (__float_as_uint(np[g].z) > wbits) | (__float_as_uint(np[g].w) > hbits);
        gone |= ((oob0 ? 1u : 0u) | (oob1 ? 2u : 0u)) << (2 * g);
        const float d0 = dist2_f32(ox, oy, np[g].x, np[g].y), d1 = dist2_f32(ox, oy, np[g].z, np[g].w);   // :151
        conf |= ((d0 < k.sep2_f ? 1u : 0u) | (d1 < k.sep2_f ? 2u : 0u)) << (2 * g);
        nmac |= ((d0 < k.nmac2_f ? 1u : 0u) | (d1 < k.nmac2_f ? 2u : 0u)) << (2 * g);
        near2 = fminf(near2, fminf(d0, d1));
      }
      if (!runs) {                                          // nobody moves: carry the positions over
        gone = conf = nmac = 0;
#pragma unroll
        for (int g = 0; g < kChunkUnits; ++g) np[g] = p[g];
      }
      if (has_env) {
        // plain store, no evict_first hint: the plane written now is the plane the NEXT step reads, and with the
        // observation stream marked evict_first a good part of its 42 MB is still in the 126 MB L2 then
        // (48.6 -> 44.9 us per step; keeping the velocities as well - plain or evict_last loads - pushes the
        // positions out again and gives the gain back)
#pragma unroll
        for (int g = 0; g < kChunkUnits; ++g) *reinterpret_cast<float4*>(pdst + g * 512) = np[g];
      }
      // The plane just read is dead when nothing can put an intruder back where it was (auto-reset): its lines -
      // largely still dirty in the L2 from the step that wrote them - are DISCARDED instead of being written back to
      // DRAM (44.9 -> 43.3 us per step).  Lanes 0, 8, 16, 24 each discard the 128 bytes
      // that they and their 7 neighbours loaded; every (tile, unit) line is read by this warp only; the address
      // carries a dependency on the loaded data so that the discard cannot overtake the loads.  The plane is written in
      // full by the next step (stream + spawn phase) before anything reads it again.
      if (a.auto_reset && (lane & 7) == 0) {
#pragma unroll
        for (int g = 0; g < kChunkUnits; ++g) {
          const uint8_t* q = psrc + g * 512 + ((__float_as_uint(np[g].x) | __float_as_uint(np[g].w)) & 0u);
          asm volatile("discard.global.L2 [%0], 128;" ::"l"(q) : "memory");
        }
      }
      if constexpr (OM != 0) {
        // observation entries -> this lane's staging row -> transposed write-out: 8 consecutive lanes store
        // the 128 contiguous bytes of ONE env's row, 4 rows per store instruction.
        uint8_t* stg = stage_smem + wib * kWarpSmem;
        float4* row = reinterpret_cast<float4*>(stg + lane * kObsRow);
#pragma unroll
        for (int g = 0; g < kChunkUnits; ++g) {
          row[2 * g] = obs_intruder_vec(k, np[g].x, np[g].y, vv[g].x, vv[g].y);
          row[2 * g + 1] = obs_intruder_vec(k, np[g].z, np[g].w, vv[g].z, vv[g].w);
        }
        __syncwarp();
        constexpr int kLanesPerEnv = kChunkIntr, kEnvsPerStore = 32 / kLanesPerEnv;
        const int sub = lane / kLanesPerEnv, chunk = lane % kLanesPerEnv;
        const uint8_t* src = stg + sub * kObsRow + chunk * 16;
        const size_t env_sub = (size_t)tile * 32 + sub;
        float* dst = reinterpret_cast<float*>(a.obs) + env_sub * (size_t)a.D + (OM == 2 ? 6 : 0) + 4 * (size_t)(i0 + chunk);
        const size_t dstep = kEnvsPerStore * (size_t)a.D;
#pragma unroll
        for (int it = 0; it < kLanesPerEnv; ++it) {
          const float4 val = *reinterpret_cast<const float4*>(src + it * kEnvsPerStore * kObsRow);
          if (env_sub + kEnvsPerStore * it < (size_t)s.B) {
            if constexpr (OM == 1) {
              stg_stream(dst + it * dstep, val, pol);
            } else {
              // own-first rows (4 N + 6 entries, the intruders from entry 6 on): an entry is 16-byte aligned in every
              // other row only (one 16-byte store there, two 8-byte stores elsewhere).  History: with every position
              // store marked evict_first, plain observation stores were faster here (the sectors that two work items
              // share got merged in the L2: 55.9 -> 52.1 us); since the position plane is kept in the L2 on purpose
              // the observation stream must not compete with it, and evict_first is the better hint again (50.1 -> 49.3).
              if ((reinterpret_cast<uintptr_t>(dst + it * dstep) & 15u) == 0) {
                stg_stream(dst + it * dstep, val, pol);
              } else {
                stg_stream2(dst + it * dstep, val.x, val.y, pol);
                stg_stream2(dst + it * dstep + 2, val.z, val.w, pol);
              }
            }
          }
        }
      } else if (has_env) {
#pragma unroll
        for (int g = 0; g < kChunkUnits; ++g) {
          Intr<FAITH> n0, n1;
          n0.px = np[g].x; n0.py = np[g].y; n0.vx = vv[g].x; n0.vy = vv[g].y;
          n1.px = np[g].z; n1.py = np[g].w; n1.vx = vv[g].z; n1.vy = vv[g].w;
          write_obs_intruder<FAITH>(a, obase, i0 + 2 * g, n0);
          write_obs_intruder<FAITH>(a, obase, i0 + 2 * g + 1, n1);
        }
      }
    }
  }
  if constexpr (FAITH) {
    if (n_here == kChunkIntr) {
      // ---- FAITHFUL, a full work item: the 8 position units and 4 velocity units are requested before any of them is
      // looked at; the f64 observation entries (32 bytes per intruder) leave through a transposed shared-memory
      // write-out - 16 consecutive lanes store the 256 contiguous bytes of ONE env's row, whole 32-byte sectors
      // (a lane storing its own 16-byte pieces 2 624 bytes apart touched 32 half-used sectors per instruction)
      fast_done = true;
      const bool stage = a.cfg.obs_kind != GCA_OBS_NONE && a.cfg.obs_kind != GCA_OBS_NEAREST && a.cfg.obs_kind != GCA_OBS_RAW6;
      double2 pq[kChunkIntr];
      float4 vq[kChunkUnits];
#pragma unroll
      for (int g = 0; g < kChunkUnits; ++g) vq[g] = ldg_stream(vsrc + g * 512, pol);
#pragma unroll
      for (int j = 0; j < kChunkIntr; ++j) {
        const float4 raw = ldg_stream(psrc + j * 512, pol);
        pq[j] = make_double2(__hiloint2double(__float_as_int(raw.y), __float_as_int(raw.x)),
                             __hiloint2double(__float_as_int(raw.w), __float_as_int(raw.z)));
      }
      const uint32_t dw = has_env ? s.dflag[flag_index(s, me, i0 >> 5)] >> (i0 & 31) : 0u;
      uint8_t* stg = stage_smem + wib * kWarpSmem;
      double2* row = reinterpret_cast<double2*>(stg + lane * kObsRow64);
#pragma unroll
      for (int j = 0; j < kChunkIntr; ++j) {
        Intr<FAITH> it;
        it.px = pq[j].x; it.py = pq[j].y;
        it.vx = (j & 1) ? vq[j >> 1].z : vq[j >> 1].x;
        it.vy = (j & 1) ? vq[j >> 1].w : vq[j >> 1].y;
        it.is64 = (dw >> j) & 1u;
        if (runs) {
          const bool oob = advance<FAITH, DRIFT>(k, it);      // :150, :153
          bool lt_sep, lt_nmac, lt_init;
          separation<FAITH>(k, ox, oy, it, lt_sep, lt_nmac, lt_init);   // :151
          gone |= (oob ? 1u : 0u) << j;
          conf |= (lt_sep ? 1u : 0u) << j;
          nmac |= (lt_nmac ? 1u : 0u) << j;
        }
        if (has_env) *reinterpret_cast<double2*>(pdst + j * 512) = make_double2(it.px, it.py);
        if (stage) {
          double o0, o1, o2, o3;
          obs_intruder_entries<FAITH>(a, it, o0, o1, o2, o3);
          row[2 * j] = make_double2(o0, o1);
          row[2 * j + 1] = make_double2(o2, o3);
        }
      }
      if (stage) {
        __syncwarp();
        const int sub = lane >> 4, piece = lane & 15;       // 16 lanes x 16 bytes = one env's 8 intruders
        const size_t row_off = (own_first(a.cfg) ? 6 : 0) + 4 * (size_t)i0;
#pragma unroll 4
        for (int it2 = 0; it2 < 16; ++it2) {
          const int e = sub + 2 * it2;
          const size_t env_e = (size_t)tile * 32 + e;
          if (env_e < (size_t)s.B) {
            const double2 val = *reinterpret_cast<const double2*>(stg + e * kObsRow64 + piece * 16);
            double* dst = reinterpret_cast<double*>(a.obs) + env_e * (size_t)a.D + row_off + 2 * (size_t)piece;
            *reinterpret_cast<double2*>(dst) = val;
          }
        }
      }
    }
  }
  if (!fast_done && has_env) {
    // ---- generic: FAITHFUL positions (f64-capable) and the ragged last work item of a tile
    uint32_t dw = 0;
    if constexpr (FAITH) dw = s.dflag[flag_index(s, me, i0 >> 5)] >> (i0 & 31);
    for (int j = 0; j < n_here; ++j) {
      const int i = i0 + j;
      Intr<FAITH> it;
      const float2 v = *reinterpret_cast<const float2*>(vsrc + (j >> 1) * 512 + (j & 1) * 8);
      it.vx = v.x; it.vy = v.y;
      if constexpr (FAITH) {
        const double2 q = *reinterpret_cast<const double2*>(psrc + j * 512);
        it.px = q.x; it.py = q.y;
        it.is64 = (dw >> j) & 1u;
      } else {
        const float2 q = *reinterpret_cast<const float2*>(psrc + (j >> 1) * 512 + (j & 1) * 8);
        it.px = q.x; it.py = q.y;
      }
      if (runs) {
        const bool oob = advance<FAITH, DRIFT>(k, it);      // :150, :153
        bool lt_sep, lt_nmac, lt_init;
        separation<FAITH>(k, ox, oy, it, lt_sep, lt_nmac, lt_init);   // :151
        gone |= (oob ? 1u : 0u) << j;
        conf |= (lt_sep ? 1u : 0u) << j;
        nmac |= (lt_nmac ? 1u : 0u) << j;
        if constexpr (!FAITH) near2 = fminf(near2, dist2_f32(ox, oy, it.px, it.py));
      }
      if constexpr (FAITH) *reinterpret_cast<double2*>(pdst + j * 512) = make_double2(it.px, it.py);
      else *reinterpret_cast<float2*>(pdst + (j >> 1) * 512 + (j & 1) * 8) = make_float2(it.px, it.py);
      write_obs_intruder<FAITH>(a, obase, i, it);
    }
  }
  // ---- record the (rare) events; i0 is a multiple of 8, so the 8 bits never straddle a word
  if (has_env) {
    const size_t fi = flag_index(s, me, i0 >> 5);
    if (gone) atomicOr(&s.ev_gone[fi], gone << (i0 & 31));
    if (conf) atomicOr(&s.ev_conf[fi], conf << (i0 & 31));
    nmac &= conf;                                           // `if dist < NMAC_dist` sits inside `if dist < minimum_separation`
    if (nmac) atomicMin(&s.ev_nmac[me], i0 + __ffs(nmac) - 1);
    if constexpr (!FAITH) {                                 // non-negative floats order like their bit patterns
      if (a.cfg.shaped_nearest && runs) atomicMin(&s.ev_near[me], __float_as_uint(near2));
    }
  }
  } while (0);
#ifdef GCA_PHASE_TIMING
  __syncthreads();
  if (threadIdx.x == 0 && blockIdx.x < 8192) g_cta[2 * blockIdx.x + 1] = gtime();
#endif
  GCA_KSTAMP_OUT(1);
}

// ------------------------------------------------------------------------------ reset / observe
template <bool FAITH, bool TAPE>
__global__ void __launch_bounds__(128) reset_kernel(const StepArgs a) {
  const DevState& s = a.s;
  const int lane = threadIdx.x & 31;
  const long long tile = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (tile >= s.T) return;
  const size_t env0 = (size_t)tile * 32;
  const bool has_env = env0 + lane < (size_t)s.B;
  const size_t me = has_env ? env0 + lane : env0;
  const bool selected = has_env && (a.mask == nullptr || a.mask[me] != 0);
  int4 cnt = make_int4(0, 0, 0, 0);
  if (has_env) cnt = s.counters[me];
  Draws<TAPE> d = make_draws<TAPE>(a, me, (uint32_t)cnt.z);
  const int nxt = (cnt.z & 1) ^ 1;                       // a reset is a tick too: it writes the other plane
  float2 pos = make_float2(0.f, 0.f);
  double2 hs = make_double2(0., 0.), vel = make_double2(0., 0.), goal = make_double2(0., 0.);
  reset_envs_warp<FAITH, TAPE>(a, env0, lane, selected, nxt, d, pos, hs, vel, goal);
  if (selected) {
    store_own_reset<FAITH>(a, me, pos, hs, vel, goal, cnt);
    cnt.z += 1;
    s.counters[me] = cnt;
    if constexpr (TAPE) a.cursor[me] = d.cur;
    if (a.done) a.done[me] = 0;
    if (a.info) a.info[me] = 0;
  }
}

// _get_ob() of the current state   PKG/SingleAircraftEnv.py:100-126; thread = env, plane reads are coalesced
template <bool FAITH>
__global__ void __launch_bounds__(128) observe_kernel(const StepArgs a) {
  const DevState& s = a.s;
  const size_t me = (size_t)blockIdx.x * 128 + threadIdx.x;
  if (me >= (size_t)s.B) return;
  const int plane = s.counters[me].z & 1;
  real_t<FAITH>* obase = obs_intruder_base<FAITH>(a, me);
  for (int i = 0; i < s.N; ++i) {
    Intr<FAITH> it;
    load_intruder<FAITH>(s, plane, me, i, it);
    write_obs_intruder<FAITH>(a, obase, i, it);
  }
  const float2 pos = s.own_pos[me];
  const double2 hs = s.own_hs[me], vel = s.own_vel[me], goal = s.goal[me];
  write_obs_own<FAITH>(a, me, pos.x, pos.y, vel.x, vel.y, s.own_vel_f32[me] != 0, hs.x, hs.y, goal.x, goal.y);
}

// GCA_OBS_NEAREST: the observation needs the n nearest of the FINAL intruder set (after respawns / resets), so it is a
// pass of its own behind the spawn kernel: thread = env, coalesced plane reads (Simulators/SingleAircraftDiscrete9HEREnv.py:106-165)
template <bool FAITH>
__global__ void __launch_bounds__(128) nearest_obs_kernel(const __grid_constant__ StepArgs a) {
  pdl_wait();
  const size_t t = (size_t)blockIdx.x * 128 + threadIdx.x;       // 4 lanes per env, 32 envs per block
  const size_t me = t >> 2;
  const bool valid = me < (size_t)a.s.B;
  if (__ballot_sync(FULL, valid) == 0u) return;
  if (a.cfg.nearest_n <= 4) write_obs_nearest<FAITH, 4>(a, valid ? me : (size_t)a.s.B - 1, (int)(t & 3), valid);
  else write_obs_nearest<FAITH, 8>(a, valid ? me : (size_t)a.s.B - 1, (int)(t & 3), valid);
}

// Simulators/SingleAircraftMCTSRandIntruderEnv.py: _update_headings (:166-174, TURN) and the six raw entries per intruder
// of _get_ob (:133-140).  Both need the FINAL intruder set of the step (after respawns / resets), so this is a pass of
// its own behind spawn_kernel, like nearest_obs_kernel.  A turn depends on (env, tick, intruder) only (Philox slot
// GCA_SLOT_TURN).  TAPE handles replay the turns inside finish_tile (draw order) and run this pass with TURN = false.
// block = 8 intruders of the 32 envs of a tile; warp = one 16-byte plane unit (intruders 2u, 2u + 1), lane = env, so
// every plane read is a whole 512-byte line.  The six entries per intruder go through shared memory and leave as the
// 8 x 24 (FAST) / 8 x 48 (FAITHFUL) contiguous bytes of each env's row - a lane storing its own entries 1952 bytes
// apart touched 32 partly used sectors per instruction and the pass was bound by L1 store sectors (first cut: 83 us).
constexpr int kTurnIntr = 8;                          // intruders per block
template <bool FAITH, bool TURN>
__global__ void __launch_bounds__(128, 16) turn_obs_kernel(const __grid_constant__ StepArgs a) {
  pdl_wait();
  using R = real_t<FAITH>;
  using V2 = typename std::conditional<FAITH, double2, float2>::type;
  constexpr int kRowV2 = 3 * kTurnIntr;               // V2 elements of one env's piece
  constexpr int kRowStride = kRowV2 + 1;              // (+ 1: conflict-free 8 / 16-byte shared accesses by lane = env)
  __shared__ V2 stage[32 * kRowStride];
  __shared__ uint16_t turn_list[32 * kTurnIntr];      // (env lane << 3 | intruder - i0) of the intruders that turn
  __shared__ int turn_count;
  const DevState& s = a.s;
  const gca_config& c = a.cfg;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int per_tile = (s.N + kTurnIntr - 1) / kTurnIntr;
  const int tile = (int)(blockIdx.x / per_tile);
  const int i0 = (int)(blockIdx.x % per_tile) * kTurnIntr;
  const size_t me = (size_t)tile * 32 + lane;
  const bool has_env = me < (size_t)s.B;
  const bool obs = c.obs_kind == GCA_OBS_RAW6;
  const bool may_turn = TURN && c.intruder_turns && s.ihs;
  const int u = i0 / 2 + wib;                          // this warp's plane unit
  if (TURN && threadIdx.x == 0) turn_count = 0;
  if (TURN) __syncthreads();
  // ---- phase 1, lane = env: plane reads, who turns, the entries as they stand
  if (has_env && 2 * u < s.N) {
    const int4 cnt = s.counters[me];
    const int plane = cnt.z & 1;
    const uint8_t* pbase = s.ipos + (size_t)plane * s.pos_plane;
    double px[2], py[2];
    if constexpr (FAITH) {
      const double2 p0 = *reinterpret_cast<const double2*>(pbase + ipos_offset(s, true, me, 2 * u));
      const double2 p1 = *reinterpret_cast<const double2*>(pbase + ipos_offset(s, true, me, 2 * u) + 512);   // unit 2u + 1
      px[0] = p0.x; py[0] = p0.y; px[1] = p1.x; py[1] = p1.y;
    } else {
      const float4 p = *reinterpret_cast<const float4*>(pbase + ipos_offset(s, false, me, 2 * u));
      px[0] = p.x; py[0] = p.y; px[1] = p.z; py[1] = p.w;
    }
    const float4 v = *reinterpret_cast<const float4*>(s.ivel + ivel_offset(s, me, 2 * u));
    const float vx[2] = {v.x, v.z}, vy[2] = {v.y, v.w};
    // one Philox block holds the p of both intruders of the unit; p < turn_prob is decided on the 53-bit integers, so
    // the ~90 % that fly on cost no f64 work.  ep_steps == 0 after a step: the env finished and was reset
    // (auto-reset) - the turns of its old intruders are moot.
    bool turn_h[2] = {false, false};
    if (may_turn && !(a.auto_reset && cnt.y == 0)) {
      const uint4 w = philox4x32_10(make_uint4(a.env_id0 + (uint32_t)me, (uint32_t)cnt.z - 1u, GCA_SLOT_TURN | (uint32_t)u, 0u),
                                    a.key0, a.key1);
      turn_h[0] = (((unsigned long long)(w.x >> 5) << 26) | (unsigned long long)(w.y >> 6)) < a.k.turn_thresh;
      turn_h[1] = (((unsigned long long)(w.z >> 5) << 26) | (unsigned long long)(w.w >> 6)) < a.k.turn_thresh;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = 2 * u + h;
      if (i >= s.N) break;
      if (turn_h[h]) turn_list[atomicAdd(&turn_count, 1)] = (uint16_t)((lane << 3) | (i - i0));
      if (obs) {
        const double2 ih = s.ihs ? s.ihs[ihs_index(s, me, i)] : make_double2(0.0, 0.0);
        V2* o = stage + lane * kRowStride + 3 * (i - i0);
        o[0] = V2{(R)px[h], (R)py[h]};
        o[1] = V2{(R)vx[h], (R)vy[h]};
        o[2] = V2{(R)ih.y, (R)ih.x};
      }
    }
  }
  if (!TURN && !obs) return;
  __syncthreads();
  // ---- phase 2, thread = one turning intruder of the block (about 26 of 256): the f64 work runs densely instead of
  // once per warp that holds a turner (97 % of them).  change_heading :332-336
  if constexpr (TURN) {
    for (int k = threadIdx.x; k < turn_count; k += 128) {
      const int e = turn_list[k] >> 3, i = i0 + (turn_list[k] & 7);
      const size_t env = (size_t)tile * 32 + e;
      Draws<false> d;
      d.k0 = a.key0; d.k1 = a.key1;
      d.env = a.env_id0 + (uint32_t)env;
      d.tick = (uint32_t)s.counters[env].z - 1u;            // the tick of the step that just ran
      double uu, unused, sn, cs;
      d.uniform2(GCA_SLOT_TURN | (uint32_t)i, 1u, uu, unused);
      // math.radians(np.random.uniform(-10, 10)): low + (high - low) * u, then * (pi / 180)
      const double raw = __dadd_rn(-c.turn_max_deg, __dmul_rn(__dadd_rn(c.turn_max_deg, c.turn_max_deg), uu));
      double2 ih = s.ihs[ihs_index(s, env, i)];
      ih.x = __dadd_rn(ih.x, __dmul_rn(raw, 3.141592653589793 / 180.0));
      gca_sincos(ih.x, &sn, &cs);
      const float nvx = (float)__dmul_rn(ih.y, cs), nvy = (float)__dmul_rn(ih.y, sn);
      s.ihs[ihs_index(s, env, i)] = ih;
      store_ivel(s, env, i, nvx, nvy);
      if (obs) {
        V2* o = stage + e * kRowStride + 3 * (i - i0);
        o[1] = V2{(R)nvx, (R)nvy};
        o[2] = V2{(R)ih.y, (R)ih.x};
      }
    }
    if (!obs) return;
    __syncthreads();
  }
  // ---- phase 3: each env's piece of the row leaves as contiguous bytes
  const int n_here = min(kTurnIntr, s.N - i0);
  const int row_v2 = 3 * n_here;                       // valid V2 elements per env
  for (int idx = threadIdx.x; idx < 32 * kRowV2; idx += 128) {
    const int e = idx / kRowV2, j = idx - e * kRowV2;
    const size_t env = (size_t)tile * 32 + e;
    if (j < row_v2 && env < (size_t)s.B) {
      R* dst = reinterpret_cast<R*>(a.obs) + env * (size_t)a.D + 6 * (size_t)i0;     // 8-byte (FAST) / 16-byte aligned
      reinterpret_cast<V2*>(dst)[j] = stage[e * kRowStride + j];
    }
  }
}

static bool has_turn_pass(const StepArgs& a) {
  return a.s.N > 0 && (a.cfg.obs_kind == GCA_OBS_RAW6 || (a.cfg.intruder_turns && a.s.ihs));
}
static unsigned turn_blocks(const DevState& s) { return (unsigned)((size_t)s.T * (size_t)((s.N + kTurnIntr - 1) / kTurnIntr)); }

// ------------------------------------------------------------------------------ launchers
// ev (nullable): 5 events recorded before / between / after the kernels of the step (gca_profile_*):
//   TAPE    0 own 1 streaming 2 finish 3 (-) 4
//   PHILOX  0 (-) 1 ownship role + streaming 2 finish + spawn phase 3 nearest / turn pass 4
template <bool FAITH, bool TAPE>
static cudaError_t launch_step_t(const StepArgs& a0, cudaStream_t st, cudaEvent_t* ev) {
  StepArgs a = a0;
  const DevState& s = a.s;
  const unsigned env_blocks = (unsigned)(((size_t)s.T * 32 + 127) / 128);
  // profiling events; inside a stream capture they must be EXTERNAL records to become event-record nodes of the graph
  // (a plain record would only be a capture-internal dependency and could not be timed)
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (ev) cudaStreamIsCapturing(st, &cap);
  auto mark = [&](int i) {
    if (!ev) return;
    if (cap == cudaStreamCaptureStatusActive) cudaEventRecordWithFlags(ev[i], st, cudaEventRecordExternal);
    else cudaEventRecord(ev[i], st);
  };
  mark(0);
  a.own_blocks = 0;
  if constexpr (TAPE) launch_pdl(step_own_kernel<FAITH, TAPE>, env_blocks, 128, st, a);
  mark(1);
  if (!TAPE && s.N == 0) {
    if constexpr (!TAPE) {
      if (s.B > (1 << 18)) launch_pdl(step_n0_kernel<FAITH, 8>, env_blocks, 128, st, a);
      else launch_pdl(step_n0_kernel<FAITH, 1>, env_blocks, 128, st, a);
    }
    mark(2);
    mark(3);
    mark(4);
    return cudaGetLastError();
  }
  if (s.N > 0) {
    const int n_chunks = (s.U + kChunkUnits - 1) / kChunkUnits;
    a.own_blocks = TAPE ? 0 : (int)(((size_t)s.T * 32 + kWarpsB * 32 - 1) / (kWarpsB * 32));   // (thread = env, blocks of the streaming kernel's size)
    const unsigned blocks = (unsigned)(((long long)s.T * n_chunks + kWarpsB - 1) / kWarpsB) + (unsigned)a.own_blocks;
    if constexpr (FAITH) {
      if (a.k.has_drift) launch_pdl(step_intruders_kernel<true, 0, true>, blocks, kWarpsB * 32, st, a);
      else launch_pdl(step_intruders_kernel<true, 0>, blocks, kWarpsB * 32, st, a);
    } else {
      const bool own_first = a.cfg.obs_kind == GCA_OBS_HER || a.cfg.obs_kind == GCA_OBS_DHER;
      const bool special = a.k.div1_ok && !a.k.has_drift;
      if (special && a.cfg.obs_kind == GCA_OBS_VECTOR) launch_pdl(step_intruders_kernel<false, 1>, blocks, kWarpsB * 32, st, a);
      else if (special && own_first) launch_pdl(step_intruders_kernel<false, 2>, blocks, kWarpsB * 32, st, a);
      else if (a.k.has_drift) launch_pdl(step_intruders_kernel<false, 0, true>, blocks, kWarpsB * 32, st, a);
      else launch_pdl(step_intruders_kernel<false, 0>, blocks, kWarpsB * 32, st, a);
    }
  }
  mark(2);
  launch_pdl(step_finish_kernel<FAITH, TAPE>, (unsigned)((s.T + 3) / 4), 128, st, a);
  mark(3);
  if (a.cfg.obs_kind == GCA_OBS_NEAREST)
    launch_pdl(nearest_obs_kernel<FAITH>, (unsigned)(((size_t)s.B + 31) / 32), 128, st, a);
  if (has_turn_pass(a)) launch_pdl(turn_obs_kernel<FAITH, !TAPE>, turn_blocks(s), 128, st, a);
  mark(4);
  return cudaGetLastError();
}

cudaError_t launch_step(bool faith, bool tape, const StepArgs& a, cudaStream_t st, cudaEvent_t* ev) {
  if (faith) return tape ? launch_step_t<true, true>(a, st, ev) : launch_step_t<true, false>(a, st, ev);
  return tape ? launch_step_t<false, true>(a, st, ev) : launch_step_t<false, false>(a, st, ev);
}

// kernels one gca_step launches for this configuration (bench.py's gpu_launches)
int step_launch_count(bool tape, int n_intruders, int obs_kind, bool turns) {
  if (!tape && n_intruders == 0) return 1 + (obs_kind == GCA_OBS_NEAREST ? 1 : 0);   // step_n0_kernel
  // TAPE: own, streaming, finish.  PHILOX: ownship role + streaming, finish + spawn phase.
  return (tape ? 2 : 1) + (n_intruders > 0 ? 1 : 0) + (obs_kind == GCA_OBS_NEAREST ? 1 : 0) +
         (n_intruders > 0 && (obs_kind == GCA_OBS_RAW6 || turns) ? 1 : 0);
}

cudaError_t launch_reset(bool faith, bool tape, const StepArgs& a, cudaStream_t st) {
  const unsigned blocks = (unsigned)((a.s.T + 3) / 4);
  if (faith) {
    if (tape) reset_kernel<true, true><<<blocks, 128, 0, st>>>(a);
    else reset_kernel<true, false><<<blocks, 128, 0, st>>>(a);
  } else {
    if (tape) reset_kernel<false, true><<<blocks, 128, 0, st>>>(a);
    else reset_kernel<false, false><<<blocks, 128, 0, st>>>(a);
  }
  if (a.cfg.obs_kind == GCA_OBS_NEAREST) return launch_observe(faith, a, st);
  if (a.cfg.obs_kind == GCA_OBS_RAW6 && a.s.N > 0) {       // the intruder entries of the reset observation
    if (faith) turn_obs_kernel<true, false><<<turn_blocks(a.s), 128, 0, st>>>(a);
    else turn_obs_kernel<false, false><<<turn_blocks(a.s), 128, 0, st>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t launch_observe(bool faith, const StepArgs& a, cudaStream_t st) {
  const unsigned blocks = (unsigned)(((size_t)a.s.B + 127) / 128);
  if (a.cfg.obs_kind == GCA_OBS_NEAREST) {
    const unsigned nb = (unsigned)(((size_t)a.s.B + 31) / 32);
    if (faith) nearest_obs_kernel<true><<<nb, 128, 0, st>>>(a);
    else nearest_obs_kernel<false><<<nb, 128, 0, st>>>(a);
  } else if (faith) observe_kernel<true><<<blocks, 128, 0, st>>>(a);
  else observe_kernel<false><<<blocks, 128, 0, st>>>(a);
  if (a.cfg.obs_kind == GCA_OBS_RAW6 && a.s.N > 0) {       // (observe_kernel wrote the ownship / goal tail)
    if (faith) turn_obs_kernel<true, false><<<turn_blocks(a.s), 128, 0, st>>>(a);
    else turn_obs_kernel<false, false><<<turn_blocks(a.s), 128, 0, st>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace gca
