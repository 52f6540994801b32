// gca_mcts.cu - the MCTS forward model of the reference as batched device-side playouts (sm_100a).
//
// Reference: Algorithms/MCTS/nodes_single.py (SingleAircraftState.move :39-100, reward :25-32,
// is_terminal_state :34-37, rollout :198-204), common.py (rollout_policy :54-55),
// config_single.py.  All arithmetic is f64 (the model works on Python floats); the quirks are
// kept: the last intruder is ignored (Q22), speed = clamp(own vy) so the throttle is inert (Q23),
// conflict and goal both use minimum_separation and there is no NMAC tier (Q24), the wall test
// is strict (Q6).
//
// Users of the model (details at each kernel):
//   mcts_playout_packed_kernel      position_sigma == 0 (the reference's setting): intruder trajectories shared by a
//                                   root's playouts, one playout per lane;
//   mcts_playout_rnd_lane_kernel    the random-intruder model up to 80 intruders and 256 playouts: one playout per lane;
//   mcts_playout_kernel<RC, RND>    every other playout launch: one warp per playout (below);
//   mcts_candidates_kernel + mcts_search_kernel   the whole UCT search of a root in one lane, trees resident in HBM;
//   mcts_move_kernel                one move() per state (the drop-in node classes, tape replay).
//
// playout kernel: one warp per playout.  What is sequential in the reference is split so that the
// expensive f64 work runs lane-parallel:
//   (1) lane f draws the heading noise of sub-frame f (Philox + Box-Muller)        - parallel
//   (2) headings are accumulated in the reference's order (h += dpsi; h += noise)    - 2 DADD / frame
//   (3) lane f evaluates sincos(h_f)                                                 - parallel
//   (4) the speed / position recurrence (speed_f = clamp(vy_{f-1})) runs as a short uniform
//       loop fed by shuffles; lane f keeps the ownship position of sub-frame f
//   (5) sub-frame loop, lanes = intruders: positions advance by repeated f64 addition exactly
//       like the reference, squared distance against the pre-squared threshold, __any_sync;
//       the loop ends at the first sub-frame with a wall / conflict / goal event.
// The kernel is bound by the FP64 pipe (about 8 DFMA-class instructions per intruder per sub-frame),
// not by HBM: a root state (2.6 KB at N = 80) is read once per playout and stays in registers.
#include <algorithm>
#include "gca_launch.h"

namespace gca {

struct MctsArgs {
  gca_mcts_config c;
  double sep2;              // min{ s : sqrt(s) >= minimum_separation }
  int n, near, L;
  int per;                  // entries per intruder of a state vector: 4 (nodes_single.py), 6 (nodes_single_randintru.py)
  // playouts
  const double* roots;
  long long n_roots;
  int playouts, depth;
  const int8_t* first_action;
  uint32_t key0, key1, root_id0;
  double* rewards;
  int8_t* first_out;
  uint8_t* flags;
  // search
  int sims;
  uint8_t* workspace;
  size_t ws_root_stride, ws_cand_off, ws_node_off;
  int32_t* best_action;
  double *child_n, *child_q;
  int32_t* child_action;
  // move
  double* states;
  const int32_t* actions;
  long long m;
  const double* tape;
  long long tape_stride;
  long long* cursor;
  int first_frame;
  int cull;                 // random_intruders playouts: drop the intruders that cannot come within the separation radius
};

__device__ __forceinline__ void mcts_uniform2(const MctsArgs& a, uint32_t root, uint32_t playout, uint32_t what,
                                              uint32_t idx, double& u0, double& u1) {
  const uint4 w = philox4x32_10(make_uint4(root, playout, what, idx), a.key0, a.key1);
  u0 = u53(w.x, w.y);
  u1 = u53(w.z, w.w);
}

// np.random.normal(0, sigma): Box-Muller cos branch of block (what, idx)
__device__ __forceinline__ double mcts_normal(const MctsArgs& a, double sigma, uint32_t root, uint32_t playout,
                                              uint32_t what, uint32_t idx) {
  if (sigma == 0.0) return 0.0;
  double u0, u1, sn, cs;
  mcts_uniform2(a, root, playout, what, idx, u0, u1);
  const double r = __dsqrt_rn(__dmul_rn(-2.0, gca_log(__dadd_rn(1.0, -u0))));
  gca_sincos(__dmul_rn(6.283185307179586, u1), &sn, &cs);
  return __dadd_rn(0.0, __dmul_rn(sigma, __dmul_rn(r, cs)));
}

// nodes_single_randintru.py:64-65: np.random.random() < 0.1 -> heading += math.radians(np.random.uniform(-10, 10)).
// Philox block (GCA_MCTS_DRAW_TURN + intruder, global sub-frame) = (p, u).  True and the heading change on a turn.
__device__ __forceinline__ bool mcts_turn(const MctsArgs& a, uint32_t root, uint32_t playout, uint32_t intruder,
                                          uint32_t gf, double& delta) {
  double p, u;
  mcts_uniform2(a, root, playout, GCA_MCTS_DRAW_TURN + intruder, gf, p, u);
  if (!(p < a.c.turn_prob)) return false;
  const double raw = __dadd_rn(-a.c.turn_max_deg, __dmul_rn(__dadd_rn(a.c.turn_max_deg, a.c.turn_max_deg), u));
  delta = __dmul_rn(raw, 3.141592653589793 / 180.0);
  return true;
}

__device__ __forceinline__ int mcts_action(const MctsArgs& a, uint32_t root, uint32_t playout, uint32_t move) {
  double u0, u1;
  mcts_uniform2(a, root, playout, GCA_MCTS_DRAW_ACTION, move, u0, u1);
  const int k = (int)__dmul_rn(9.0, u0);
  return k > 8 ? 8 : k;
}

__device__ __forceinline__ double clamp_speed(const gca_mcts_config& c, double vy) {
  const double m = c.max_speed < vy ? c.max_speed : vy;       // min(state[-5], max_speed)
  return m > c.min_speed ? m : c.min_speed;                   // max(min_speed, .)
}

__device__ __forceinline__ double shfl_f64(double v, int src) {
  return __shfl_sync(FULL, v, src);
}

// the action of a playout's move at `depth`: the caller's first action where one is given (>= 0), else rollout_policy's
__device__ __forceinline__ int playout_action(const MctsArgs& a, long long pid, uint32_t root, uint32_t playout, int depth) {
  if (depth == 0 && a.first_action && a.first_action[pid] >= 0) return a.first_action[pid];
  return mcts_action(a, root, playout, (uint32_t)depth);
}

__device__ __forceinline__ double lane_reward(int flags, double ox, double oy, double gx, double gy) {
  if (flags & (GCA_MCTS_WALL | GCA_MCTS_CONFLICT)) return 0.0;
  if (flags & GCA_MCTS_GOAL) return 1.0;
  const double dx = __dadd_rn(ox, -gx), dy = __dadd_rn(oy, -gy);
  const double dist = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
  return __dadd_rn(1.0, -__ddiv_rn(dist, 1200.0));
}

__device__ __forceinline__ void store_playout(const MctsArgs& a, long long pid, int first, int flags, double reward) {
  a.rewards[pid] = reward;
  if (a.first_out) a.first_out[pid] = (int8_t)first;
  if (a.flags) a.flags[pid] = (uint8_t)flags;
}

// The random-intruder model (nodes_single_randintru.py) without position / speed noise (a.cull): every aircraft moves at
// most its speed per sub-frame (an intruder: its root velocity until it first turns, then `speed` along its heading; the
// ownship: clamp(...) <= max_speed).  An intruder further away at the root than both reaches plus the separation radius
// can never raise the conflict flag in the playout, and nothing else of it is observable (reward and flags are the only
// outputs): it is dropped.  The survivors keep their index - the draws of intruder i are addressed by i - so the playout
// is bit-identical to the one that simulates all N (what the oracle does); typically ~10 of 80 remain.
// One warp: the six entries of the kept intruders of root state st (ownship entries at own) go to dst, their indices to
// idx; returns how many.  Without a.cull every intruder is kept.
__device__ __forceinline__ int cull_intruders(const MctsArgs& a, const double* st, const double* own, int lane, double* dst,
                                              int* idx) {
  const gca_mcts_config& c = a.c;
  const double frames = (double)a.depth * (double)c.simulate_frame;
  const double own_reach = fmax(fabs(c.max_speed), fabs(c.min_speed)) * frames;
  int n_eff = 0;
  for (int base = 0; base < a.near; base += 32) {
    const int i = base + lane;
    double v[6] = {0., 0., 0., 0., 0., 0.};
    bool keep = false;
    if (i < a.near) {
#pragma unroll
      for (int q = 0; q < 6; ++q) v[q] = st[6 * i + q];
      const double dx = v[0] - own[0], dy = v[1] - own[1];
      const double reach = fmax(sqrt(v[2] * v[2] + v[3] * v[3]), fabs(v[4])) * frames;
      keep = !a.cull || !(sqrt(dx * dx + dy * dy) > own_reach + reach + c.minimum_separation + 2.0);   // (NaN: kept)
    }
    const uint32_t mask = __ballot_sync(FULL, keep);
    const int at = n_eff + __popc(mask & ((1u << lane) - 1u));
    if (keep) {
#pragma unroll
      for (int q = 0; q < 6; ++q) dst[6 * at + q] = v[q];
      idx[at] = i;
    }
    n_eff += __popc(mask);
  }
  return n_eff;
}

constexpr int kMctsWarps = 4;
constexpr int kMaxRounds = 4;       // intruder rounds held in registers (N - 1 <= 128); larger N uses the generic path
static_assert(kMaxRounds == 4, "launch_mcts_playouts dispatches on 1..4 rounds");

// RC > 0: intruder rounds in registers; RC == 0: intruders live in shared memory (any N).
// RND (with RC == 0): the model of nodes_single_randintru.py - six entries per intruder, every intruder may turn after
// its advance, the ownship speed is a state of its own (clamped on itself, :73-75).
template <int RC, bool RND = false>
__global__ void __launch_bounds__(kMctsWarps * 32) mcts_playout_kernel(const MctsArgs a) {
  static_assert(!(RND && RC != 0), "the random-intruder model keeps its intruders in shared memory");
  constexpr int PER = RND ? 6 : 4;
  extern __shared__ double mcts_smem[];
  const gca_mcts_config& c = a.c;
  const int lane = threadIdx.x & 31;
  const int warp_in_block = threadIdx.x >> 5;
  const long long pid = (long long)blockIdx.x * kMctsWarps + warp_in_block;
  const long long total = a.n_roots * a.playouts;
  if (pid >= total) return;
  const long long r_idx = pid / a.playouts;
  const uint32_t playout = (uint32_t)(pid - r_idx * a.playouts);
  const uint32_t root = a.root_id0 + (uint32_t)r_idx;
  const double* st = a.roots + r_idx * a.L;
  const double* own = st + a.per * a.n;

  // ---- intruders: lane i + 32 r holds (x, y, vx, vy)
  double ix[RC > 0 ? RC : 1], iy[RC > 0 ? RC : 1], ivx[RC > 0 ? RC : 1], ivy[RC > 0 ? RC : 1];
  // RC == 0 only: this warp's intruders, then (RND) their original indices - what the Philox draws are addressed by
  const size_t warp_doubles = (size_t)PER * a.near + (RND ? ((size_t)a.near + 1) / 2 : 0);
  double* sm = mcts_smem + (size_t)warp_in_block * warp_doubles;
  int* sidx = reinterpret_cast<int*>(sm + (size_t)PER * a.near);
  int n_eff = a.near;                                               // intruders this playout simulates
  (void)sidx;
  if constexpr (RC > 0) {
#pragma unroll
    for (int r = 0; r < RC; ++r) {
      const int i = r * 32 + lane;
      const bool v = i < a.near;
      const double2 p = v ? reinterpret_cast<const double2*>(st)[2 * i] : make_double2(0., 0.);
      const double2 w = v ? reinterpret_cast<const double2*>(st)[2 * i + 1] : make_double2(0., 0.);
      ix[r] = p.x; iy[r] = p.y; ivx[r] = w.x; ivy[r] = w.y;
    }
  } else if constexpr (RND) {
    n_eff = cull_intruders(a, st, own, lane, sm, sidx);
    __syncwarp();
  } else {
    for (int j = lane; j < PER * a.near; j += 32) sm[j] = st[j];
    __syncwarp();
  }
  double ox = own[0], oy = own[1], vy_prev = own[3], speed = own[4], heading = own[5];
  const double gx = own[6], gy = own[7];
  (void)speed;

  const int F = c.simulate_frame;
  int flags = 0, first = -1;
  int depth = 0;
  // ---- one move() per iteration; sub-frames handled in chunks of 32 lanes
  while (!(flags || depth == a.depth)) {
    const int act = playout_action(a, pid, root, playout, depth);
    if (first < 0) first = act;
    const double d_heading = __dmul_rn((double)(act / 3 - 1), c.d_heading);
    const double accel = __dmul_rn((double)(act % 3 - 1), c.d_speed);
    (void)accel;
    for (int f0 = 0; f0 < F && !flags; f0 += 32) {
      const int nf = min(32, F - f0);
      const uint32_t gf = (uint32_t)(depth * F + f0 + lane);
      // (1) noises of sub-frame f0 + lane
      double nh = 0.0, nsp = 0.0;
      if (lane < nf) {
        nh = mcts_normal(a, c.heading_sigma, root, playout, GCA_MCTS_DRAW_HEADING, gf);
        nsp = mcts_normal(a, c.speed_sigma, root, playout, GCA_MCTS_DRAW_SPEED, gf);
      }
      // (2) headings in the reference's order
      double my_h = 0.0;
      for (int f = 0; f < nf; ++f) {
        heading = __dadd_rn(heading, d_heading);                      // state[-3] += d_heading
        heading = __dadd_rn(heading, shfl_f64(nh, f));                // state[-3] += normal(0, heading_sigma)
        if (lane == f) my_h = heading;
      }
      // (3) sincos of each sub-frame's heading
      double sn = 0.0, cs = 1.0;
      if (lane < nf) gca_sincos(my_h, &sn, &cs);
      // (4) speed / position recurrence; lane f keeps the ownship position of sub-frame f
      double my_ox = 0.0, my_oy = 0.0;
      for (int f = 0; f < nf; ++f) {
        double sp;
        if constexpr (RND) sp = clamp_speed(c, __dadd_rn(speed, accel));   // state[-4] += a; state[-4] = clamp(state[-4])
        else sp = clamp_speed(c, vy_prev);                            // state[-4] = clamp(state[-5])  (Q23)
        sp = __dadd_rn(sp, shfl_f64(nsp, f));                         // += normal(0, speed_sigma)
        speed = sp;
        const double vx = __dmul_rn(sp, shfl_f64(cs, f)), vy = __dmul_rn(sp, shfl_f64(sn, f));
        ox = __dadd_rn(ox, vx);
        oy = __dadd_rn(oy, vy);
        vy_prev = vy;
        if (lane == f) { my_ox = ox; my_oy = oy; }
      }
      // per-sub-frame ownship events, evaluated lane-parallel
      const bool wall = lane < nf && (!(0.0 < my_ox && my_ox < c.window_width) || !(0.0 < my_oy && my_oy < c.window_height));
      bool goal = false;
      if (lane < nf) {
        const double dx = __dadd_rn(my_ox, -gx), dy = __dadd_rn(my_oy, -gy);
        goal = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;   // metric(own, goal) < minimum_separation
      }
      const uint32_t wall_mask = __ballot_sync(FULL, wall), goal_mask = __ballot_sync(FULL, goal);
      // (5) intruders, sub-frame by sub-frame, until the first event
      int f_end = nf;
      for (int f = 0; f < nf; ++f) {
        const uint32_t gfu = (uint32_t)(depth * F + f0 + f);
        const double fx = shfl_f64(my_ox, f), fy = shfl_f64(my_oy, f);
        bool hit = false;
        if constexpr (RC > 0) {
#pragma unroll
          for (int r = 0; r < RC; ++r) {
            const int i = r * 32 + lane;
            if (i < a.near) {
              const double npx = mcts_normal(a, c.position_sigma, root, playout, GCA_MCTS_DRAW_INTRUDER + (uint32_t)i, 2 * gfu);
              const double npy = mcts_normal(a, c.position_sigma, root, playout, GCA_MCTS_DRAW_INTRUDER + (uint32_t)i, 2 * gfu + 1);
              ix[r] = __dadd_rn(ix[r], __dadd_rn(ivx[r], npx));      // x += vx + normal(0, position_sigma)
              iy[r] = __dadd_rn(iy[r], __dadd_rn(ivy[r], npy));
              const double dx = __dadd_rn(ix[r], -fx), dy = __dadd_rn(iy[r], -fy);
              hit |= __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;
            }
          }
        } else {
          for (int i = lane; i < n_eff; i += 32) {
            uint32_t ii = (uint32_t)i;                                // the intruder's own index addresses its draws
            if constexpr (RND) ii = (uint32_t)sidx[i];
            const double npx = mcts_normal(a, c.position_sigma, root, playout, GCA_MCTS_DRAW_INTRUDER + ii, 2 * gfu);
            const double npy = mcts_normal(a, c.position_sigma, root, playout, GCA_MCTS_DRAW_INTRUDER + ii, 2 * gfu + 1);
            const double x = __dadd_rn(sm[PER * i], __dadd_rn(sm[PER * i + 2], npx));
            const double y = __dadd_rn(sm[PER * i + 1], __dadd_rn(sm[PER * i + 3], npy));
            sm[PER * i] = x;
            sm[PER * i + 1] = y;
            if constexpr (RND) {                                      // the turn follows the advance (:64-71)
              double delta;
              if (mcts_turn(a, root, playout, ii, gfu, delta)) {
                double tsn, tcs;
                const double h = __dadd_rn(sm[6 * i + 5], delta);
                gca_sincos(h, &tsn, &tcs);
                sm[6 * i + 2] = __dmul_rn(sm[6 * i + 4], tcs);
                sm[6 * i + 3] = __dmul_rn(sm[6 * i + 4], tsn);
                sm[6 * i + 5] = h;
              }
            }
            const double dx = __dadd_rn(x, -fx), dy = __dadd_rn(y, -fy);
            hit |= __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;
          }
        }
        const bool conflict = __any_sync(FULL, hit);
        // order inside a sub-frame: wall, then conflict, then goal (nodes_single.py:80-98)
        if ((wall_mask >> f) & 1u) flags = GCA_MCTS_WALL;
        else if (conflict) flags = GCA_MCTS_CONFLICT;
        else if ((goal_mask >> f) & 1u) flags = GCA_MCTS_GOAL;
        if (flags) {
          f_end = f + 1;
          break;
        }
      }
      // the ownship state of the playout is the one of the last executed sub-frame
      ox = shfl_f64(my_ox, f_end - 1);
      oy = shfl_f64(my_oy, f_end - 1);
    }
    ++depth;
  }
  if (lane == 0) store_playout(a, pid, first, flags, lane_reward(flags, ox, oy, gx, gy));
}

// ---- position_sigma == 0 (config_single.py:27, the reference's setting): the intruders of the model move on
// trajectories that depend on nothing but the root - x_f = x_{f-1} + (vx + 0.0), the same f64 additions for every
// playout of that root - and the ownship cannot move further than (gf + 1) * max_speed from its root position (ox0, oy0)
// by global sub-frame gf when speed_sigma == 0 (speed = clamp(vy) in [min_speed, max_speed], Q23).  One sub-frame of an
// intruder's trajectory: advances (x, y) through sub-frame gf and returns whether the ownship could reach it there (the
// margins cover the rounding of the bound).
__device__ __forceinline__ bool advance_in_reach(const gca_mcts_config& c, double ox0, double oy0, int gf, double vx,
                                                 double vy, double& x, double& y) {
  x = __dadd_rn(x, vx);
  y = __dadd_rn(y, vy);
  if (c.speed_sigma != 0.0) return true;
  const double vmax = fmax(fabs(c.min_speed), fabs(c.max_speed));
  const double reach = c.minimum_separation + (double)(gf + 1) * vmax * 1.000001 + 0.5;
  const double dx = x - ox0, dy = y - oy0;
  return !(dx * dx + dy * dy >= reach * reach);
}

// COMPACT: cnt[gf] .. cnt[gf + 1] delimit the sub-frame's candidates in one packed list (the search workspace);
// otherwise cnt[gf] candidates at cand[gf * near] (the shared-memory layout of the packed playout kernel)
template <bool COMPACT = false>
__device__ __forceinline__ int lane_move(const MctsArgs& a, const int* __restrict__ cnt, const double2* __restrict__ cand,
                                         uint32_t root, uint32_t sim, int depth, int act, double gx, double gy,
                                         double& ox, double& oy, double& vy_prev, double& heading);

// The lanes of a CTA are the playouts of R consecutive roots laid end to end (5 roots x 100 playouts = 500 of 512
// lanes); a root with more than kPackThreads playouts runs alone (R = 1) in slices of kPackThreads playouts, a CTA per
// slice (blockIdx.y), each slice rebuilding its root's candidate lists.  Per depth:
//   phase 1 (thread = (root, intruder)): advance every intruder of the R roots through the depth's sub-frames from where
//           the previous depth left it (running position in shared memory, the same chain of additions) and, per
//           sub-frame, list (exact f64 position) those the ownship could reach;
//   phase 2 (thread = playout): the playout's move of that depth runs in one lane - Philox / Box-Muller / sincos per
//           sub-frame in the reference's order, wall test, exact distance test against the sub-frame's candidates only
//           (uniform shared-memory reads), goal test - with no shuffles and no idle lanes in the scalar part.
// Same arithmetic per playout as mcts_playout_kernel, so the results are bit-identical; at N = 80 the 79 x 30 distance
// tests of a playout collapse to ~45.  The candidate lists exist for one depth at a time (simulate_frame sub-frames:
// 12.8 KB per root at N = 80), so two CTAs fit an SM.
constexpr int kPackThreads = 512;             // 2 CTAs x 512 threads x 64 registers fill the register file
constexpr int kPackMaxRoots = 8;

__global__ void __launch_bounds__(kPackThreads, 2) mcts_playout_packed_kernel(const MctsArgs a, const int R) {
  extern __shared__ __align__(16) uint8_t mcts_sh[];
  const gca_mcts_config& c = a.c;
  const int F = c.simulate_frame, near = a.near;
  // layout: cnt [R][F] ints | xs [R][near] double2 | cand [R][F][near] double2
  int* cnt = reinterpret_cast<int*>(mcts_sh);
  double2* xs = reinterpret_cast<double2*>(mcts_sh + (((size_t)R * F * 4 + 15) & ~(size_t)15));
  double2* cand = xs + (size_t)R * near;
  const long long r0 = (long long)blockIdx.x * R;
  const int r_here = (int)min((long long)R, a.n_roots - r0);
  const int q = threadIdx.x, rl = q / a.playouts, p = q - rl * a.playouts + (int)(blockIdx.y * blockDim.x);
  const bool active = rl < r_here && p < a.playouts;
  const long long r_idx = r0 + (active ? rl : 0);
  const uint32_t root = a.root_id0 + (uint32_t)r_idx;
  const double* own = a.roots + r_idx * a.L + a.per * a.n;
  const double gx = own[6], gy = own[7];
  const long long pid = r_idx * a.playouts + p;
  double ox = own[0], oy = own[1], vy_prev = own[3], heading = own[5];
  int flags = 0, first = -1;
  for (int depth = 0; depth < a.depth; ++depth) {
    for (int f = threadIdx.x; f < r_here * F; f += blockDim.x) cnt[f] = 0;
    __syncthreads();
    // ---- phase 1 of this depth: thread = (root, intruder)
    for (int idx = threadIdx.x; idx < r_here * near; idx += blockDim.x) {
      const int jr = idx / near, i = idx - jr * near;
      const double* st = a.roots + (r0 + jr) * a.L;
      const double* jo = st + a.per * a.n;
      const double ox0 = jo[0], oy0 = jo[1];
      const double2 v0 = reinterpret_cast<const double2*>(st)[2 * i + 1];
      double2 pos = depth == 0 ? reinterpret_cast<const double2*>(st)[2 * i] : xs[(size_t)jr * near + i];
      double x = pos.x, y = pos.y;
      const double vx = __dadd_rn(v0.x, 0.0), vy = __dadd_rn(v0.y, 0.0);     // vx + normal(0, 0) :54-57
      for (int f = 0; f < F; ++f) {
        if (advance_in_reach(c, ox0, oy0, depth * F + f, vx, vy, x, y))
          cand[((size_t)jr * F + f) * near + atomicAdd(&cnt[jr * F + f], 1)] = make_double2(x, y);
      }
      xs[(size_t)jr * near + i] = make_double2(x, y);
    }
    __syncthreads();
    // ---- phase 2 of this depth: lane = playout (lane_move indexes the lists by global sub-frame: shift the bases)
    if (active && !flags) {
      const int act = playout_action(a, pid, root, (uint32_t)p, depth);
      if (first < 0) first = act;
      flags = lane_move(a, cnt + (rl - depth) * F, cand + (ptrdiff_t)(rl - depth) * F * near, root, (uint32_t)p, depth, act, gx, gy,
                        ox, oy, vy_prev, heading);
    }
    __syncthreads();
  }
  if (active) store_playout(a, pid, first, flags, lane_reward(flags, ox, oy, gx, gy));
}

// ---- the random-intruder model (nodes_single_randintru.py), one playout per LANE.  In mcts_playout_kernel<0, true> a
// warp runs one playout with lane = intruder (after the exact cull ~10 of 32 lanes) or lane = sub-frame (10 of 32) -
// a third of every instruction does work.  Here the lanes of a CTA are the playouts of R consecutive roots laid end
// to end; a warp per root culls the root's intruders once into shared memory (the survivors and their original
// indices - the draws of intruder i are addressed by i), and every lane then runs its playout sequentially on a
// private copy of the survivors (thread-local arrays: position, velocity and heading change per playout) - the same
// operations in the same order per playout and intruder as the warp kernel, so the same bits.
// measured at 100 playouts per root: 256 threads (2 roots, 200 of 224 lanes), 3 CTAs per SM at 79 registers: 4.3e8
// rollouts/s; 512 x 1 (112 registers) 3.6e8, 512 x 2 / 128 x 8 (64, spills) 3.8e8
constexpr int kLaneThreads = 256;
constexpr int kLaneMinBlocks = 3;
constexpr int kLaneMaxRoots = 8;
constexpr int kLaneMaxNear = 80;              // thread-local arrays; larger models take the warp-per-playout kernel

__global__ void __launch_bounds__(kLaneThreads, kLaneMinBlocks) mcts_playout_rnd_lane_kernel(const MctsArgs a, const int R) {
  extern __shared__ __align__(16) uint8_t mcts_sh[];
  const gca_mcts_config& c = a.c;
  const int F = c.simulate_frame, near = a.near;
  // layout: neff [R] ints (padded to 16 B) | sidx [R][near] ints | base [R][near][6] doubles
  int* neff = reinterpret_cast<int*>(mcts_sh);
  int* sidx = neff + 16;
  double* base = reinterpret_cast<double*>(mcts_sh + (((size_t)(16 + (size_t)R * near) * 4 + 15) & ~(size_t)15));
  const long long r0 = (long long)blockIdx.x * R;
  const int r_here = (int)min((long long)R, a.n_roots - r0);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  // ---- cull, a warp per root
  for (int jr = wib; jr < r_here; jr += n_warps) {
    const double* st = a.roots + (r0 + jr) * a.L;
    const int n_eff = cull_intruders(a, st, st + a.per * a.n, lane, base + (size_t)jr * near * 6, sidx + jr * near);
    if (lane == 0) neff[jr] = n_eff;
  }
  __syncthreads();
  // ---- lane = playout
  const int q = threadIdx.x, rl = q / a.playouts, p = q - rl * a.playouts;
  if (rl >= r_here) return;
  const long long r_idx = r0 + rl;
  const uint32_t root = a.root_id0 + (uint32_t)r_idx, playout = (uint32_t)p;
  const double* own = a.roots + r_idx * a.L + a.per * a.n;
  const long long pid = r_idx * a.playouts + p;
  const int n_eff = neff[rl];
  const int* my_idx = sidx + rl * near;
  const double* my_base = base + (size_t)rl * near * 6;
  double X[kLaneMaxNear], Y[kLaneMaxNear], VX[kLaneMaxNear], VY[kLaneMaxNear], H[kLaneMaxNear];
  for (int j = 0; j < n_eff; ++j) {
    X[j] = my_base[6 * j]; Y[j] = my_base[6 * j + 1]; VX[j] = my_base[6 * j + 2]; VY[j] = my_base[6 * j + 3];
    H[j] = my_base[6 * j + 5];
  }
  constexpr int kTurnQueue = 8;
  int turn_j[kTurnQueue], n_turns = 0;
  double turn_d[kTurnQueue];
  auto apply_turn = [&](int j, double delta) {
    double tsn, tcs;
    const double h = __dadd_rn(H[j], delta);
    gca_sincos(h, &tsn, &tcs);
    VX[j] = __dmul_rn(my_base[6 * j + 4], tcs);
    VY[j] = __dmul_rn(my_base[6 * j + 4], tsn);
    H[j] = h;
  };
  double ox = own[0], oy = own[1], speed = own[4], heading = own[5];
  const double gx = own[6], gy = own[7];
  int flags = 0, first = -1;
  for (int depth = 0; depth < a.depth && !flags; ++depth) {
    const int act = playout_action(a, pid, root, playout, depth);
    if (first < 0) first = act;
    const double d_heading = __dmul_rn((double)(act / 3 - 1), c.d_heading);
    const double accel = __dmul_rn((double)(act % 3 - 1), c.d_speed);
    for (int f = 0; f < F; ++f) {
      const uint32_t gf = (uint32_t)(depth * F + f);
      const double nh = mcts_normal(a, c.heading_sigma, root, playout, GCA_MCTS_DRAW_HEADING, gf);
      const double nsp = mcts_normal(a, c.speed_sigma, root, playout, GCA_MCTS_DRAW_SPEED, gf);
      heading = __dadd_rn(heading, d_heading);                        // state[-3] += d_heading
      heading = __dadd_rn(heading, nh);                               // state[-3] += normal(0, heading_sigma)
      double sn, cs;
      gca_sincos(heading, &sn, &cs);
      double sp = clamp_speed(c, __dadd_rn(speed, accel));            // state[-4] += a; state[-4] = clamp(state[-4])
      sp = __dadd_rn(sp, nsp);                                        // += normal(0, speed_sigma)
      speed = sp;
      ox = __dadd_rn(ox, __dmul_rn(sp, cs));
      oy = __dadd_rn(oy, __dmul_rn(sp, sn));
      // order inside a sub-frame: wall, then conflict, then goal (nodes_single.py:80-98); what the intruders do in a
      // sub-frame that ends the playout is not observable
      if (!(0.0 < ox && ox < c.window_width) || !(0.0 < oy && oy < c.window_height)) { flags = GCA_MCTS_WALL; break; }
      bool hit = false;
      for (int j = 0; j < n_eff; ++j) {
        const uint32_t ii = (uint32_t)my_idx[j];                      // the intruder's own index addresses its draws
        const double npx = mcts_normal(a, c.position_sigma, root, playout, GCA_MCTS_DRAW_INTRUDER + ii, 2 * gf);
        const double npy = mcts_normal(a, c.position_sigma, root, playout, GCA_MCTS_DRAW_INTRUDER + ii, 2 * gf + 1);
        const double x = __dadd_rn(X[j], __dadd_rn(VX[j], npx));
        const double y = __dadd_rn(Y[j], __dadd_rn(VY[j], npy));
        X[j] = x;
        Y[j] = y;
        // the turn follows the advance (:64-71) and touches nothing but this intruder's velocity and heading, which the
        // NEXT sub-frame reads: the (rare, 10 %) turns of a sub-frame are queued and made after the loop, where the lanes
        // that have one run the sincos together instead of one or two lanes at a time inside the loop
        double delta;
        if (mcts_turn(a, root, playout, ii, gf, delta)) {
          if (n_turns == kTurnQueue) {                                // (queue full: make the oldest now)
            --n_turns;
            apply_turn(turn_j[n_turns], turn_d[n_turns]);
          }
          turn_j[n_turns] = j;
          turn_d[n_turns] = delta;
          ++n_turns;
        }
        const double dx = __dadd_rn(x, -ox), dy = __dadd_rn(y, -oy);
        hit |= __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;
      }
      while (n_turns > 0) {
        --n_turns;
        apply_turn(turn_j[n_turns], turn_d[n_turns]);
      }
      if (hit) { flags = GCA_MCTS_CONFLICT; break; }
      const double dx = __dadd_rn(ox, -gx), dy = __dadd_rn(oy, -gy);
      if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2) { flags = GCA_MCTS_GOAL; break; }
    }
  }
  store_playout(a, pid, first, flags, lane_reward(flags, ox, oy, gx, gy));
}

// ------------------------------------------------------------------------------ device-resident UCT search
// MCTS(root).best_action(simulations, search_depth) (search_single.py:8-22; tree_policy / expand / best_child /
// backpropagate: common.py:47-52, nodes_single.py:188-210) for a batch of roots, position_sigma == 0.  Because the
// intruders of the model then follow root-only trajectories and a non-terminal node of depth d has executed exactly
// d * simulate_frame sub-frames, a tree node needs only the ownship (x, y, vy, heading): 80 bytes per node.
//   mcts_candidates_kernel: CTA per root - phase 1 of the playout kernel, candidate lists written to the workspace;
//   mcts_search_kernel:     lane per root - the search is sequential in its simulations, and 32 independent roots
//                           per warp keep every lane busy: selection (UCT in f64 with the shared log), expansion
//                           (untried actions popped from the end, Q27), rollout, back-propagation.
// Draws: Philox keyed (seed; root id, simulation index, kind, global sub-frame) - simulation s of a root is
// "playout" s of the playout kernels.  Bit-exact against gca_oracle_mcts_search_philox.
struct __align__(16) TreeNode {
  double ox, oy, vy, heading;
  double q;
  int n;
  short parent;
  signed char depth, flags, action, untried, n_children, pad;
  short children[9];
};
static_assert(sizeof(TreeNode) == 80, "tree node layout");

// simulate_frame sub-frames of move(action) from global sub-frame depth * F (nodes_single.py:39-100); returns the flags.
// One lane runs the whole move, sub-frame by sub-frame.  (Batching the state-independent noise / sincos chains of
// several sub-frames for instruction-level parallelism was measured: 2 at a time -5 %, 5 at a time -25 % - the extra
// registers cost more occupancy than the parallel chains return.)
template <bool COMPACT>
__device__ __forceinline__ int lane_move(const MctsArgs& a, const int* __restrict__ cnt, const double2* __restrict__ cand,
                                         uint32_t root, uint32_t sim, int depth, int act, double gx, double gy,
                                         double& ox, double& oy, double& vy_prev, double& heading) {
  const gca_mcts_config& c = a.c;
  const int F = c.simulate_frame;
  const double d_heading = __dmul_rn((double)(act / 3 - 1), c.d_heading);
  // COMPACT (global memory, one lane per root): the list bounds and the first four candidates of sub-frame f + 1 are
  // requested while sub-frame f computes - two dependent round trips per sub-frame otherwise.  The slots behind a
  // sub-frame's last candidate are inside the root's list area (read and ignored).
  int e0 = 0, e1 = 0;
  double2 q[4] = {};
  if constexpr (COMPACT) {
    e0 = cnt[depth * F];
    e1 = cnt[depth * F + 1];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = cand[e0 + j];
  }
  for (int f = 0; f < F; ++f) {
    const int gf = depth * F + f;
    int e2 = e1;
    double2 qn[4] = {};
    if constexpr (COMPACT) {
      if (f + 1 < F) {
        e2 = cnt[gf + 2];
#pragma unroll
        for (int j = 0; j < 4; ++j) qn[j] = cand[e1 + j];
      }
    }
    const double nh = mcts_normal(a, c.heading_sigma, root, sim, GCA_MCTS_DRAW_HEADING, (uint32_t)gf);
    const double nsp = mcts_normal(a, c.speed_sigma, root, sim, GCA_MCTS_DRAW_SPEED, (uint32_t)gf);
    double sp = clamp_speed(c, vy_prev);                              // state[-4] = clamp(state[-5])  (Q23)
    sp = __dadd_rn(sp, nsp);
    heading = __dadd_rn(heading, d_heading);                          // state[-3] += d_heading
    heading = __dadd_rn(heading, nh);                                 // state[-3] += normal(0, heading_sigma)
    double sn, cs;
    gca_sincos(heading, &sn, &cs);
    const double vx = __dmul_rn(sp, cs), vy = __dmul_rn(sp, sn);
    ox = __dadd_rn(ox, vx);
    oy = __dadd_rn(oy, vy);
    vy_prev = vy;
    if (!(0.0 < ox && ox < c.window_width) || !(0.0 < oy && oy < c.window_height)) return GCA_MCTS_WALL;
    bool hit = false;
    const double2* cf = COMPACT ? cand + e0 : cand + (size_t)gf * a.near;
    const int nc = COMPACT ? e1 - e0 : cnt[gf];
    if constexpr (COMPACT) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double dx = __dadd_rn(q[j].x, -ox), dy = __dadd_rn(q[j].y, -oy);
        hit |= (j < nc) & (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2);
      }
      for (int k = 4; k < nc; ++k) {                                  // (rarely more than four)
        const double2 r = cf[k];
        const double dx = __dadd_rn(r.x, -ox), dy = __dadd_rn(r.y, -oy);
        hit |= __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;
      }
      e0 = e1;
      e1 = e2;
#pragma unroll
      for (int j = 0; j < 4; ++j) q[j] = qn[j];
    } else {
      for (int k = 0; k < nc; ++k) {
        const double2 q = cf[k];
        const double dx = __dadd_rn(q.x, -ox), dy = __dadd_rn(q.y, -oy);
        hit |= __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;
      }
    }
    if (hit) return GCA_MCTS_CONFLICT;
    const double dx = __dadd_rn(ox, -gx), dy = __dadd_rn(oy, -gy);
    if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2) return GCA_MCTS_GOAL;
  }
  return 0;
}

// intruder trajectories of one root -> per-sub-frame candidate lists, PACKED: ends[0] = 0 and ends[f + 1] = end of
// sub-frame f's candidates in `cand` (so ends[f] is where they start).  Two passes over the same deterministic
// trajectories: count, exclusive scan, place.  Packed because the search reads them one LANE per root: with the
// [sub-frame][near] layout of the playout kernels every sub-frame of every root sat in a cache line of its own (38 KB
// per root at N = 80 for ~45 candidates); now a root's lists are ~1 KB, contiguous.
template <bool PLACE>
__device__ __forceinline__ void walk_candidates(const MctsArgs& a, const double* st, int TF, int* ends, double2* cand, int tid,
                                                int nthreads) {
  const gca_mcts_config& c = a.c;
  const double* own = st + a.per * a.n;
  const double ox0 = own[0], oy0 = own[1];
  for (int i = tid; i < a.near; i += nthreads) {
    const double2 p0 = reinterpret_cast<const double2*>(st)[2 * i];
    const double2 v0 = reinterpret_cast<const double2*>(st)[2 * i + 1];
    double x = p0.x, y = p0.y;
    const double vx = __dadd_rn(v0.x, 0.0), vy = __dadd_rn(v0.y, 0.0);       // vx + normal(0, 0) :54-57
    for (int f = 0; f < TF; ++f) {
      if (advance_in_reach(c, ox0, oy0, f, vx, vy, x, y)) {
        const int at = atomicAdd(&ends[f + 1], 1);          // count, or (PLACE) the sub-frame's fill pointer
        if (PLACE) cand[at] = make_double2(x, y);
      }
    }
  }
}

__global__ void __launch_bounds__(128) mcts_candidates_kernel(const MctsArgs a) {
  const int TF = a.depth * a.c.simulate_frame;
  uint8_t* ws = a.workspace + (size_t)blockIdx.x * a.ws_root_stride;
  int* ends = reinterpret_cast<int*>(ws);                                     // [TF + 1]
  double2* cand = reinterpret_cast<double2*>(ws + a.ws_cand_off);
  const double* st = a.roots + (long long)blockIdx.x * a.L;
  for (int f = threadIdx.x; f <= TF; f += 128) ends[f] = 0;
  __syncthreads();
  walk_candidates<false>(a, st, TF, ends, cand, threadIdx.x, 128);            // ends[f + 1] = count of sub-frame f
  __syncthreads();
  if (threadIdx.x == 0) {                                                     // -> where sub-frame f's candidates start
    int run = 0;
    for (int f = 0; f < TF; ++f) {
      const int n = ends[f + 1];
      ends[f + 1] = run;
      run += n;
    }
  }
  __syncthreads();
  walk_candidates<true>(a, st, TF, ends, cand, threadIdx.x, 128);             // fill pointers end at the sub-frame's end
}

__global__ void __launch_bounds__(128) mcts_search_kernel(const MctsArgs a) {
  const long long r_idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r_idx >= a.n_roots) return;
  const uint32_t root = a.root_id0 + (uint32_t)r_idx;
  const double* own = a.roots + r_idx * a.L + a.per * a.n;
  uint8_t* ws = a.workspace + (size_t)r_idx * a.ws_root_stride;
  const int* cnt = reinterpret_cast<const int*>(ws);
  const double2* cand = reinterpret_cast<const double2*>(ws + a.ws_cand_off);
  TreeNode* nodes = reinterpret_cast<TreeNode*>(ws + a.ws_node_off);
  const double gx = own[6], gy = own[7];
  const int D = a.depth;

  TreeNode rt{};
  rt.ox = own[0]; rt.oy = own[1]; rt.vy = own[3]; rt.heading = own[5];
  rt.parent = -1; rt.action = -1; rt.untried = 9;
  nodes[0] = rt;
  int count = 1;

  auto best_child = [&](int v, double c_param) -> int {              // common.py:47-52, np.argmax: first maximum
    const TreeNode& nv = nodes[v];
    const double lg2 = __dmul_rn(2.0, gca_log((double)nv.n));
    int best = -1;
    double best_w = 0.0;
    // the children's statistics are requested together (each sits in a cache line of its own: one round trip instead
    // of one per child), then scored in order
    const int nch = nv.n_children;
    int cidx[9], cvis[9];
    double cq[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      cidx[k] = k < nch ? nv.children[k] : 0;
      cvis[k] = nodes[cidx[k]].n;
      cq[k] = nodes[cidx[k]].q;
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      if (k < nch) {
        const double cn = (double)cvis[k];
        const double w = __dadd_rn(__ddiv_rn(cq[k], cn), __dmul_rn(c_param, __dsqrt_rn(__ddiv_rn(lg2, cn))));
        if (best < 0 || w > best_w) { best = cidx[k]; best_w = w; }
      }
    }
    return best;
  };

  // One loop iteration = at most one model move per lane.  A lane that finished a simulation back-propagates, selects
  // and (lazily) starts the next one in the same iteration, so the 32 roots of a warp execute lane_move together
  // whatever simulation / phase each of them is in (the simulations of ONE root stay strictly sequential).
  int s = 0, v = 0, flags = 0, depth = 0;
  bool expand = false, running = false;
  double ox = 0.0, oy = 0.0, vy = 0.0, heading = 0.0;
  while (s < a.sims) {
    if (!running) {
      // tree_policy (search_single.py:16-22): walk down by UCT until a node with an untried action (or a terminal one)
      v = 0;
      expand = false;
      while (!(nodes[v].flags || nodes[v].depth == D)) {
        if (nodes[v].untried > 0) { expand = true; break; }
        v = best_child(v, 1.4);
      }
      ox = nodes[v].ox; oy = nodes[v].oy; vy = nodes[v].vy; heading = nodes[v].heading;
      flags = nodes[v].flags; depth = nodes[v].depth;
      running = true;
    }
    if (!(flags || depth == D)) {
      // the expansion move (action popped from the end, nodes_single.py:188-193) and the rollout moves (random actions,
      // :198-204) are the same model step
      int act;
      if (expand) act = --nodes[v].untried;
      else act = mcts_action(a, root, (uint32_t)s, (uint32_t)depth);
      flags = lane_move<true>(a, cnt, cand, root, (uint32_t)s, depth, act, gx, gy, ox, oy, vy, heading);
      ++depth;
      if (expand) {                                                   // the new child: the state after this one move
        TreeNode ch{};
        ch.ox = ox; ch.oy = oy; ch.vy = vy; ch.heading = heading;
        ch.flags = (signed char)flags; ch.parent = (short)v; ch.depth = (signed char)depth; ch.action = (signed char)act;
        ch.untried = 9;
        nodes[count] = ch;
        nodes[v].children[nodes[v].n_children++] = (short)count;
        v = count++;
        expand = false;
      }
    }
    if (flags || depth == D) {
      const double reward = lane_reward(flags, ox, oy, gx, gy);
      for (int u = v; u >= 0; u = nodes[u].parent) {                  // backpropagate  nodes_single.py:206-210
        nodes[u].n += 1;
        nodes[u].q = __dadd_rn(nodes[u].q, reward);
      }
      running = false;
      ++s;
    }
  }
  const int b = best_child(0, 0.0);
  a.best_action[r_idx] = b >= 0 ? nodes[b].action : -1;
  for (int k = 0; k < 9; ++k) {
    const bool has = k < nodes[0].n_children;
    const int ci = has ? nodes[0].children[k] : 0;
    if (a.child_n) a.child_n[r_idx * 9 + k] = has ? (double)nodes[ci].n : 0.0;
    if (a.child_q) a.child_q[r_idx * 9 + k] = has ? nodes[ci].q : 0.0;
    if (a.child_action) a.child_action[r_idx * 9 + k] = has ? nodes[ci].action : -1;
  }
}

// SingleAircraftState.move for m independent states, one thread each, in the reference's own
// sequential order (used by the drop-in node classes and by the tape-replay parity tests).
__global__ void __launch_bounds__(128) mcts_move_kernel(const MctsArgs a) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= a.m) return;
  const gca_mcts_config& c = a.c;
  double* st = a.states + k * a.L;
  double* own = st + a.per * a.n;
  const int act = a.actions[k];
  const double d_heading = __dmul_rn((double)(act / 3 - 1), c.d_heading);
  const double accel = __dmul_rn((double)(act % 3 - 1), c.d_speed);
  const bool tape = a.tape != nullptr;
  const double* tp = tape ? a.tape + k * a.tape_stride : nullptr;
  long long cur = tape ? a.cursor[k] : 0;
  const uint32_t root = a.root_id0 + (uint32_t)k;
  int flags = 0;
  for (int f = 0; f < c.simulate_frame; ++f) {
    const uint32_t gf = (uint32_t)(a.first_frame + f);
    for (int i = 0; i < a.near; ++i) {
      double* it = st + a.per * i;
      const double nx = tape ? tp[cur++] : mcts_normal(a, c.position_sigma, root, 0u, GCA_MCTS_DRAW_INTRUDER + (uint32_t)i, 2 * gf);
      it[0] = __dadd_rn(it[0], __dadd_rn(it[2], nx));
      const double ny = tape ? tp[cur++] : mcts_normal(a, c.position_sigma, root, 0u, GCA_MCTS_DRAW_INTRUDER + (uint32_t)i, 2 * gf + 1);
      it[1] = __dadd_rn(it[1], __dadd_rn(it[3], ny));
      if (c.random_intruders) {                       // nodes_single_randintru.py:64-71
        double delta = 0.0;
        bool turn;
        if (tape) {
          turn = tp[cur++] < c.turn_prob;             // np.random.random()
          if (turn) delta = __dmul_rn(tp[cur++], 3.141592653589793 / 180.0);   // math.radians(np.random.uniform(-10, 10))
        } else {
          turn = mcts_turn(a, root, 0u, (uint32_t)i, gf, delta);
        }
        if (turn) {
          double tsn, tcs;
          const double h = __dadd_rn(it[5], delta);
          gca_sincos(h, &tsn, &tcs);
          it[2] = __dmul_rn(it[4], tcs);
          it[3] = __dmul_rn(it[4], tsn);
          it[5] = h;
        }
      }
    }
    own[4] = __dadd_rn(own[4], accel);
    own[4] = clamp_speed(c, c.random_intruders ? own[4] : own[3]);     // (:74 clamps the speed; nodes_single.py:60 reads vy, Q23)
    own[4] = __dadd_rn(own[4], tape ? tp[cur++] : mcts_normal(a, c.speed_sigma, root, 0u, GCA_MCTS_DRAW_SPEED, gf));
    own[5] = __dadd_rn(own[5], d_heading);
    own[5] = __dadd_rn(own[5], tape ? tp[cur++] : mcts_normal(a, c.heading_sigma, root, 0u, GCA_MCTS_DRAW_HEADING, gf));
    double sn, cs;
    gca_sincos(own[5], &sn, &cs);
    const double vx = __dmul_rn(own[4], cs), vy = __dmul_rn(own[4], sn);
    own[0] = __dadd_rn(own[0], vx);
    own[1] = __dadd_rn(own[1], vy);
    own[2] = vx;
    own[3] = vy;
    const double ox = own[0], oy = own[1];
    if (!(0.0 < ox && ox < c.window_width) || !(0.0 < oy && oy < c.window_height)) {
      flags = GCA_MCTS_WALL;
      break;
    }
    bool conflict = false;
    for (int i = 0; i < a.near && !conflict; ++i) {
      const double dx = __dadd_rn(st[a.per * i], -ox), dy = __dadd_rn(st[a.per * i + 1], -oy);
      conflict = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2;
    }
    if (conflict) {
      flags = GCA_MCTS_CONFLICT;
      break;
    }
    const double dx = __dadd_rn(ox, -own[6]), dy = __dadd_rn(oy, -own[7]);
    if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < a.sep2) {
      flags = GCA_MCTS_GOAL;
      break;
    }
  }
  a.flags[k] = (uint8_t)flags;
  if (tape) a.cursor[k] = cur;
}

static MctsArgs mcts_base(const gca_mcts_config* cfg, int n) {
  MctsArgs a{};
  a.c = *cfg;
  a.sep2 = sq_threshold<double>(cfg->minimum_separation);
  a.n = n;
  a.per = cfg->random_intruders ? 6 : 4;
  a.L = a.per * n + 8;
  // (len - 9) // 4: the last intruder is ignored (Q22); nodes_single_randintru.py:47 has (len - 8) // 6 = N
  a.near = cfg->random_intruders ? n : (a.L >= 9 ? (a.L - 9) / 4 : 0);
  return a;
}

cudaError_t launch_mcts_playouts(const gca_mcts_config* cfg, int n, const double* roots, long long n_roots, int playouts,
                                 int depth, const int8_t* first_action, uint64_t seed, uint32_t root_id0,
                                 double* rewards, int8_t* first_out, uint8_t* flags, cudaStream_t st) {
  MctsArgs a = mcts_base(cfg, n);
  a.roots = roots; a.n_roots = n_roots; a.playouts = playouts; a.depth = depth; a.first_action = first_action;
  a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.root_id0 = root_id0;
  a.rewards = rewards; a.first_out = first_out; a.flags = flags;
  const long long total = n_roots * playouts;
  if (total <= 0) return cudaSuccess;
  const unsigned blocks = (unsigned)((total + kMctsWarps - 1) / kMctsWarps);
  if (cfg->random_intruders) {                // every playout moves its own intruders
    a.cull = cfg->position_sigma == 0.0 && cfg->speed_sigma == 0.0;
    if (a.near <= kLaneMaxNear && playouts <= kLaneThreads) {
      // one playout per lane, several roots per CTA (mcts_playout_rnd_lane_kernel)
      const int R = (int)std::min<long long>(std::min<long long>(kLaneMaxRoots, kLaneThreads / playouts), n_roots);
      const size_t lsm = (((size_t)(16 + (size_t)R * a.near) * 4 + 15) & ~(size_t)15) + sizeof(double) * 6 * (size_t)R * (size_t)a.near;
      const unsigned threads = (unsigned)(((long long)R * playouts + 31) / 32 * 32);
      cudaError_t e = cudaFuncSetAttribute(mcts_playout_rnd_lane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm);
      if (e != cudaSuccess) return e;
      mcts_playout_rnd_lane_kernel<<<(unsigned)((n_roots + R - 1) / R), threads, lsm, st>>>(a, R);
      return cudaGetLastError();
    }
    const size_t smem = sizeof(double) * kMctsWarps * (6 * (size_t)a.near + ((size_t)a.near + 1) / 2);
    cudaError_t e = cudaFuncSetAttribute(mcts_playout_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    mcts_playout_kernel<0, true><<<blocks, kMctsWarps * 32, smem, st>>>(a);
    return cudaGetLastError();
  }
  if (cfg->position_sigma == 0.0) {
    // intruder trajectories shared by a root's playouts: several roots per CTA, or one root in slices of kPackThreads
    // playouts (mcts_playout_packed_kernel)
    const size_t F = (size_t)cfg->simulate_frame;
    auto pack_smem = [&](int r) { return (((size_t)r * F * 4 + 15) & ~(size_t)15) + sizeof(double2) * (size_t)r * (size_t)a.near * (1 + F); };
    int R = (int)std::min<long long>(std::min(kPackMaxRoots, std::max(1, kPackThreads / playouts)), n_roots);
    while (R > 1 && 2 * pack_smem(R) > 200 * 1024) --R;      // two CTAs per SM
    const unsigned slices = (unsigned)((playouts + kPackThreads - 1) / kPackThreads);
    if (pack_smem(R) <= 200 * 1024 && slices <= 65535) {     // (65535: the largest gridDim.y)
      const unsigned threads = (unsigned)((std::min((long long)R * playouts, (long long)kPackThreads) + 31) / 32 * 32);
      cudaError_t e = cudaFuncSetAttribute(mcts_playout_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pack_smem(R));
      if (e != cudaSuccess) return e;
      mcts_playout_packed_kernel<<<dim3((unsigned)((n_roots + R - 1) / R), slices), threads, pack_smem(R), st>>>(a, R);
      return cudaGetLastError();
    }
  }
  const int rounds = (a.near + 31) / 32;
  switch (rounds) {
    case 0:
    case 1: mcts_playout_kernel<1><<<blocks, kMctsWarps * 32, 0, st>>>(a); break;
    case 2: mcts_playout_kernel<2><<<blocks, kMctsWarps * 32, 0, st>>>(a); break;
    case 3: mcts_playout_kernel<3><<<blocks, kMctsWarps * 32, 0, st>>>(a); break;
    case 4: mcts_playout_kernel<4><<<blocks, kMctsWarps * 32, 0, st>>>(a); break;
    default: {
      const size_t smem = sizeof(double) * kMctsWarps * 4 * (size_t)a.near;
      cudaError_t e = cudaFuncSetAttribute(mcts_playout_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      mcts_playout_kernel<0><<<blocks, kMctsWarps * 32, smem, st>>>(a);
    }
  }
  return cudaGetLastError();
}

static void search_layout(int near, long long tf, int sims, size_t* cand_off, size_t* node_off, size_t* stride) {
  *cand_off = (((size_t)tf + 1) * 4 + 15) & ~(size_t)15;         // ends[tf + 1], then the packed candidates (worst case tf * near)
  *node_off = *cand_off + sizeof(double2) * ((size_t)tf * (size_t)near + 3);   // (+ 3: lane_move reads candidates four at a time)
  *stride = *node_off + sizeof(TreeNode) * ((size_t)sims + 1);
}

size_t mcts_search_workspace_bytes(const gca_mcts_config* cfg, int n, long long n_roots, int sims, int depth) {
  MctsArgs a = mcts_base(cfg, n);
  size_t co, no, st;
  search_layout(a.near, (long long)depth * cfg->simulate_frame, sims, &co, &no, &st);
  return st * (size_t)(n_roots > 0 ? n_roots : 0);
}

cudaError_t launch_mcts_search(const gca_mcts_config* cfg, int n, const double* roots, long long n_roots, int sims,
                               int depth, uint64_t seed, uint32_t root_id0, void* workspace, int32_t* best_action,
                               double* child_n, double* child_q, int32_t* child_action, cudaStream_t st) {
  MctsArgs a = mcts_base(cfg, n);
  a.roots = roots; a.n_roots = n_roots; a.sims = sims; a.depth = depth;
  a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.root_id0 = root_id0;
  a.workspace = static_cast<uint8_t*>(workspace);
  search_layout(a.near, (long long)depth * cfg->simulate_frame, sims, &a.ws_cand_off, &a.ws_node_off, &a.ws_root_stride);
  a.best_action = best_action; a.child_n = child_n; a.child_q = child_q; a.child_action = child_action;
  if (n_roots <= 0) return cudaSuccess;
  mcts_candidates_kernel<<<(unsigned)n_roots, 128, 0, st>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  mcts_search_kernel<<<(unsigned)((n_roots + 31) / 32), 32, 0, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_mcts_move(const gca_mcts_config* cfg, int n, double* states, const int32_t* actions, uint8_t* flags,
                             long long m, const double* tape, long long tape_stride, long long* cursor, uint64_t seed,
                             uint32_t id0, int first_frame, cudaStream_t st) {
  MctsArgs a = mcts_base(cfg, n);
  a.states = states; a.actions = actions; a.flags = flags; a.m = m;
  a.tape = tape; a.tape_stride = tape_stride; a.cursor = cursor;
  a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.root_id0 = id0; a.first_frame = first_frame;
  if (m <= 0) return cudaSuccess;
  mcts_move_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(a);
  return cudaGetLastError();
}

}  // namespace gca
