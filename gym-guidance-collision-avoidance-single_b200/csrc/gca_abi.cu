// gca_abi.cu - the C ABI of include/gca.h: handle lifetime, argument checking, state
// marshalling and the host-buffer (end-to-end) path.  No exception crosses the boundary.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <limits>
#include <map>
#include <mutex>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "gca.h"
#include "gca_launch.h"

using namespace gca;

namespace {
thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  return fail(GCA_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define GCA_CUDA(call)                                   \
  do {                                                   \
    cudaError_t e_ = (call);                             \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call);  \
  } while (0)
}  // namespace

struct gca_env {
  int device = 0, mode = 0, draws = 0;
  gca_config cfg{};
  Derived k{};
  uint64_t seed = 0;
  uint32_t env_id0 = 0;
  DevState s{};
  int D = 0;
  // host path (gca_step_host[_begin / _wait] / gca_reset_host): compute stream, download stream, two sets of
  // device-side buffers and the events that order them
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  void* d_actions[2] = {nullptr, nullptr};
  gca_out d_out[2] = {};
  cudaEvent_t ev_step[2] = {nullptr, nullptr}, ev_copy[2] = {nullptr, nullptr};
  unsigned long long host_begun = 0, host_waited = 0;
  std::vector<void*> allocs;
  // gca_profile_*
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;     // 5 per recorded step
  std::vector<cudaEvent_t> prof_pool;       // recycled
};

namespace {
size_t real_size(const gca_env* e) { return e->mode == GCA_MODE_FAITHFUL ? sizeof(double) : sizeof(float); }

int check_config(const gca_config* c) {
  if (!c) return fail(GCA_ERR_INVALID, "config is NULL");
  if (c->action_kind < GCA_ACT_DISCRETE9 || c->action_kind > GCA_ACT_DISCRETE3_HEADING) return fail(GCA_ERR_INVALID, "bad action_kind");
  if (c->obs_kind < GCA_OBS_VECTOR || c->obs_kind > GCA_OBS_RAW6) return fail(GCA_ERR_INVALID, "bad obs_kind");
  if (c->intruder_turns && !(c->turn_prob >= 0.0 && c->turn_prob <= 1.0 && c->turn_max_deg >= 0.0))
    return fail(GCA_ERR_INVALID, "intruder_turns needs 0 <= turn_prob <= 1 and turn_max_deg >= 0");
  if (c->obs_kind == GCA_OBS_NEAREST && (c->nearest_n < 1 || c->nearest_n > 8 || !(c->ob_diagonal > 0)))
    return fail(GCA_ERR_INVALID, "GCA_OBS_NEAREST needs 1 <= nearest_n <= 8 and a positive ob_diagonal");
  if (c->wall_kind < GCA_WALL_NONE || c->wall_kind > GCA_WALL_PENALTY) return fail(GCA_ERR_INVALID, "bad wall_kind");
  if (!(c->window_width > 0) || !(c->window_height > 0)) return fail(GCA_ERR_INVALID, "window must be positive");
  return GCA_OK;
}

template <typename T>
int dev_alloc(gca_env* e, T** p, size_t count) {
  void* q = nullptr;
  GCA_CUDA(cudaMalloc(&q, (count ? count : 1) * sizeof(T)));
  GCA_CUDA(cudaMemset(q, 0, (count ? count : 1) * sizeof(T)));
  e->allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return GCA_OK;
}

// cached exhaustive check that the one-correction division is exact for divisor d
bool div1_exact(float d) {
  static std::mutex mu;
  static std::map<float, bool> cache;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(d);
  if (it != cache.end()) return it->second;
  const bool ok = d > 0 && std::isfinite(d) && gca_div1_is_exact(d) != 0;
  cache[d] = ok;
  return ok;
}

Derived derive(const gca_config& c) {
  Derived k{};
  k.sep2_f = sq_threshold<float>((float)c.minimum_separation);
  k.nmac2_f = sq_threshold<float>((float)c.nmac_dist);
  k.init2_f = sq_threshold<float>((float)c.initial_min_dist);
  k.sep2_d = sq_threshold<double>(c.minimum_separation);
  k.nmac2_d = sq_threshold<double>(c.nmac_dist);
  k.init2_d = sq_threshold<double>(c.initial_min_dist);
  k.goal2_d = sq_threshold<double>(c.goal_radius);
  k.win_w = (float)c.window_width;
  k.win_h = (float)c.window_height;
  k.ob_w = (float)c.ob_window_width;
  k.ob_h = (float)c.ob_window_height;
  k.inv_ob_w = 1.0f / k.ob_w;
  k.inv_ob_h = 1.0f / k.ob_h;
  k.ms = (float)c.max_speed;
  k.den = (float)(c.max_speed * 2);
  k.inv_den = 1.0f / k.den;
  k.div1_ok = div1_exact(k.ob_w) && div1_exact(k.ob_h) && div1_exact(k.den);
  k.dv_w = c.ob_window_width;
  k.dv_h = c.ob_window_height;
  k.dv_speed = c.ob_max_speed - c.ob_min_speed;
  k.dv_2pi = 2.0 * 3.141592653589793;
  k.dv_vel = c.max_speed * 2.0;
  k.dv_shape = 1200.0;
  k.rc_w = 1.0 / k.dv_w; k.rc_h = 1.0 / k.dv_h; k.rc_speed = 1.0 / k.dv_speed;
  k.rc_2pi = 1.0 / k.dv_2pi; k.rc_vel = 1.0 / k.dv_vel; k.rc_shape = 1.0 / k.dv_shape;
  k.ddiv_ok = gca_div_f64_divisor_ok(k.dv_w) && gca_div_f64_divisor_ok(k.dv_h) && gca_div_f64_divisor_ok(k.dv_speed) &&
              gca_div_f64_divisor_ok(k.dv_2pi) && gca_div_f64_divisor_ok(k.dv_vel) && gca_div_f64_divisor_ok(k.dv_shape);
  k.drift_f = (float)c.position_drift;
  k.has_drift = c.position_drift != 0.0 ? 1 : 0;
  k.turn_thresh = c.turn_prob > 0.0 ? (unsigned long long)std::ceil(std::ldexp(c.turn_prob < 1.0 ? c.turn_prob : 1.0, 53)) : 0ull;
  return k;
}

bool keeps_ihs(const gca_config& c) { return c.intruder_turns != 0 || c.obs_kind == GCA_OBS_RAW6; }

StepArgs make_args(const gca_env* e, const void* actions, const gca_tape* tape, const gca_out* out, int auto_reset) {
  StepArgs a{};
  a.s = e->s;
  a.cfg = e->cfg;
  a.k = e->k;
  a.actions = actions;
  if (tape) {
    a.tape = tape->values;
    a.tape_stride = tape->stride;
    a.cursor = reinterpret_cast<long long*>(tape->cursor);
  }
  a.key0 = (uint32_t)e->seed;
  a.key1 = (uint32_t)(e->seed >> 32);
  a.env_id0 = e->env_id0;
  a.D = e->D;
  a.auto_reset = auto_reset;
  if (out) {
    a.obs = out->obs; a.achieved = out->achieved; a.desired = out->desired;
    a.reward = out->reward; a.done = out->done; a.info = out->info;
    a.nearest = out->nearest;
  }
  return a;
}

int check_out(const gca_env* e, const gca_out* out, bool need_reward) {
  if (!out) return fail(GCA_ERR_INVALID, "out is NULL");
  if (e->cfg.obs_kind != GCA_OBS_NONE && !out->obs) return fail(GCA_ERR_INVALID, "out->obs is NULL");
  const bool her = e->cfg.obs_kind == GCA_OBS_HER || e->cfg.obs_kind == GCA_OBS_DHER || e->cfg.obs_kind == GCA_OBS_NEAREST;
  if (her && (!out->achieved || !out->desired)) return fail(GCA_ERR_INVALID, "HER kinds need achieved/desired buffers");
  if (need_reward && (!out->reward || !out->done || !out->info)) return fail(GCA_ERR_INVALID, "reward/done/info buffers are NULL");
  return GCA_OK;
}

int check_tape(const gca_env* e, const gca_tape* tape) {
  if (e->draws == GCA_DRAWS_TAPE && (!tape || !tape->values || !tape->cursor))
    return fail(GCA_ERR_INVALID, "handle was created with GCA_DRAWS_TAPE: a tape is required");
  return GCA_OK;
}

// host copies of the tile-planar intruder planes (gca_get_state / gca_set_state)
struct HostPlanes {
  std::vector<uint8_t> pos, vel;      // pos: both planes
  std::vector<uint32_t> cf, df;
  std::vector<int4> cnt;
  std::vector<double2> hs;            // (heading, speed) plane, handles that keep it
  int download(const DevState& s, bool faith) {
    if (s.ihs) {
      hs.resize((size_t)s.T * (size_t)s.N * 32);
      GCA_CUDA(cudaMemcpy(hs.data(), s.ihs, hs.size() * sizeof(double2), cudaMemcpyDeviceToHost));
    }
    pos.resize(2 * s.pos_plane);
    vel.resize(vel_plane_bytes(s));
    cf.resize(flag_plane_words(s));
    df.resize(faith ? flag_plane_words(s) : 1);
    cnt.resize((size_t)s.B);
    GCA_CUDA(cudaMemcpy(pos.data(), s.ipos, pos.size(), cudaMemcpyDeviceToHost));
    GCA_CUDA(cudaMemcpy(vel.data(), s.ivel, vel.size(), cudaMemcpyDeviceToHost));
    GCA_CUDA(cudaMemcpy(cf.data(), s.cflag, cf.size() * 4, cudaMemcpyDeviceToHost));
    if (faith) GCA_CUDA(cudaMemcpy(df.data(), s.dflag, df.size() * 4, cudaMemcpyDeviceToHost));
    GCA_CUDA(cudaMemcpy(cnt.data(), s.counters, cnt.size() * sizeof(int4), cudaMemcpyDeviceToHost));
    return GCA_OK;
  }
  int upload(const DevState& s, bool faith) {
    if (s.ihs) GCA_CUDA(cudaMemcpy(s.ihs, hs.data(), hs.size() * sizeof(double2), cudaMemcpyHostToDevice));
    GCA_CUDA(cudaMemcpy(s.ipos, pos.data(), pos.size(), cudaMemcpyHostToDevice));
    GCA_CUDA(cudaMemcpy(s.ivel, vel.data(), vel.size(), cudaMemcpyHostToDevice));
    GCA_CUDA(cudaMemcpy(s.cflag, cf.data(), cf.size() * 4, cudaMemcpyHostToDevice));
    if (faith) GCA_CUDA(cudaMemcpy(s.dflag, df.data(), df.size() * 4, cudaMemcpyHostToDevice));
    GCA_CUDA(cudaMemcpy(s.counters, cnt.data(), cnt.size() * sizeof(int4), cudaMemcpyHostToDevice));
    return GCA_OK;
  }
  // env b's current position plane (gca_device.cuh: tick & 1)
  uint8_t* plane_of(const DevState& s, size_t b) { return pos.data() + (size_t)(cnt[b].z & 1) * s.pos_plane; }
};
}  // namespace

extern "C" {

int gca_abi_version(void) { return GCA_ABI_VERSION; }

const char* gca_last_error(void) { return g_err.c_str(); }

int gca_obs_dim(const gca_config* cfg, int n) {
  if (!cfg) return fail(GCA_ERR_INVALID, "config is NULL");
  switch (cfg->obs_kind) {
    case GCA_OBS_VECTOR:
    case GCA_OBS_RAW: return 4 * n + 8;
    case GCA_OBS_HER:
    case GCA_OBS_DHER: return 4 * n + 6;
    case GCA_OBS_NEAREST: return 4 + 5 * cfg->nearest_n;
    case GCA_OBS_RAW6: return 6 * n + 8;
    default: return 0;
  }
}

int gca_create(const gca_config* cfg, int n_envs, int n_intruders, int mode, int draws, int device, uint64_t seed,
               uint32_t env_id0, gca_env** out) {
  if (!out) return fail(GCA_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (int rc = check_config(cfg)) return rc;
  if (n_envs <= 0 || n_intruders < 0 || n_intruders > 4096) return fail(GCA_ERR_INVALID, "n_envs must be > 0 and 0 <= n_intruders <= 4096");
  if (cfg->obs_kind == GCA_OBS_NEAREST && n_intruders <= cfg->nearest_n)   // np.argpartition(dist_array, Config.n) raises otherwise
    return fail(GCA_ERR_INVALID, "GCA_OBS_NEAREST needs more intruders than nearest_n");
  if (mode != GCA_MODE_FAITHFUL && mode != GCA_MODE_FAST) return fail(GCA_ERR_INVALID, "bad mode");
  if (draws != GCA_DRAWS_TAPE && draws != GCA_DRAWS_PHILOX) return fail(GCA_ERR_INVALID, "bad draws");
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess || count <= 0)
    return fail(GCA_ERR_CUDA, std::string("no usable CUDA device (libgca has no CPU path): ") +
                                  (ce != cudaSuccess ? cudaGetErrorString(ce) : "device count is 0"));
  if (device < 0 || device >= count) return fail(GCA_ERR_INVALID, "device index out of range");
  GCA_CUDA(cudaSetDevice(device));
  gca_env* e = new (std::nothrow) gca_env();
  if (!e) return fail(GCA_ERR_ALLOC, "out of host memory");
  e->device = device; e->mode = mode; e->draws = draws; e->cfg = *cfg; e->k = derive(*cfg); e->seed = seed; e->env_id0 = env_id0;
  e->D = gca_obs_dim(cfg, n_intruders);
  DevState& s = e->s;
  s.B = n_envs; s.N = n_intruders;
  plane_layout(s, mode == GCA_MODE_FAITHFUL);
  const size_t B = (size_t)n_envs;
  int rc = GCA_OK;
  if (!rc) rc = dev_alloc(e, &s.own_pos, B);
  if (!rc) rc = dev_alloc(e, &s.own_hs, B);
  if (!rc) rc = dev_alloc(e, &s.own_vel, B);
  if (!rc) rc = dev_alloc(e, &s.own_vel_f32, B);
  if (!rc) rc = dev_alloc(e, &s.goal, B);
  if (!rc) rc = dev_alloc(e, &s.counters, B);
  if (!rc) rc = dev_alloc(e, &s.ipos, 2 * s.pos_plane);
  if (!rc) rc = dev_alloc(e, &s.own_b, (size_t)s.T * 32);
  if (!rc) rc = dev_alloc(e, &s.ev_conf, flag_plane_words(s));
  if (!rc) rc = dev_alloc(e, &s.ev_gone, flag_plane_words(s));
  if (!rc) rc = dev_alloc(e, &s.ev_nmac, (size_t)s.T * 32);
  if (!rc) rc = dev_alloc(e, &s.ev_near, (size_t)s.T * 32);
  if (!rc) rc = dev_alloc(e, &s.pre, (size_t)s.T * 32);
  if (!rc) rc = dev_alloc(e, &s.step_seq, 1);
  if (!rc) rc = dev_alloc(e, &s.error_flag, 1);
  if (!rc) rc = dev_alloc(e, &s.ivel, vel_plane_bytes(s));
  if (!rc) rc = dev_alloc(e, &s.cflag, flag_plane_words(s));
  if (!rc) rc = dev_alloc(e, &s.dflag, mode == GCA_MODE_FAITHFUL ? flag_plane_words(s) : 1);
  if (!rc && keeps_ihs(*cfg) && n_intruders > 0) rc = dev_alloc(e, &s.ihs, (size_t)s.T * (size_t)s.N * 32);
  if (!rc) {
    // the event words are consumed AND cleared by the finish of every step (PHILOX handles): they start out clear
    std::vector<int> none((size_t)s.T * 32, INT_MAX);
    std::vector<uint32_t> inf((size_t)s.T * 32, 0x7f800000u);
    if (cudaMemcpy(s.ev_nmac, none.data(), none.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(s.ev_near, inf.data(), inf.size() * sizeof(uint32_t), cudaMemcpyHostToDevice) != cudaSuccess)
      rc = fail(GCA_ERR_CUDA, "initialising the event words failed");
  }
  if (rc) {
    gca_destroy(e);
    return rc;
  }
  *out = e;
  return GCA_OK;
}

int gca_destroy(gca_env* e) {
  if (!e) return GCA_OK;
  cudaSetDevice(e->device);
  for (void* p : e->allocs) cudaFree(p);
  for (cudaEvent_t ev : e->prof_events) cudaEventDestroy(ev);
  for (cudaEvent_t ev : e->prof_pool) cudaEventDestroy(ev);
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  for (int i = 0; i < 2; ++i) {
    if (e->ev_step[i]) cudaEventDestroy(e->ev_step[i]);
    if (e->ev_copy[i]) cudaEventDestroy(e->ev_copy[i]);
  }
  delete e;
  return GCA_OK;
}

int gca_set_seed(gca_env* e, uint64_t seed) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  e->seed = seed;
  return GCA_OK;
}

int gca_set_config(gca_env* e, const gca_config* cfg) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (int rc = check_config(cfg)) return rc;
  if (gca_obs_dim(cfg, e->s.N) != e->D) return fail(GCA_ERR_STATE, "obs_kind change would alter the observation size");
  if (keeps_ihs(*cfg) && !e->s.ihs && e->s.N > 0)
    return fail(GCA_ERR_STATE, "the handle was created without per-intruder (heading, speed) state");
  e->cfg = *cfg;
  e->k = derive(*cfg);
  return GCA_OK;
}

int gca_reset(gca_env* e, const uint8_t* mask, const gca_tape* tape, const gca_out* out, void* stream) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (int rc = check_out(e, out, false)) return rc;
  if (int rc = check_tape(e, tape)) return rc;
  GCA_CUDA(cudaSetDevice(e->device));
  StepArgs a = make_args(e, nullptr, tape, out, 0);
  a.mask = mask;
  GCA_CUDA(launch_reset(e->mode == GCA_MODE_FAITHFUL, e->draws == GCA_DRAWS_TAPE, a, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_step(gca_env* e, const void* actions, const gca_tape* tape, int auto_reset, const gca_out* out, void* stream) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (!actions) return fail(GCA_ERR_INVALID, "actions is NULL");
  if (int rc = check_out(e, out, true)) return rc;
  if (int rc = check_tape(e, tape)) return rc;
  GCA_CUDA(cudaSetDevice(e->device));
  const StepArgs a = make_args(e, actions, tape, out, auto_reset);
  cudaEvent_t* ev = nullptr;
  cudaEvent_t evs[5];
  if (e->profiling) {
    for (int i = 0; i < 5; ++i) {
      if (!e->prof_pool.empty()) {
        evs[i] = e->prof_pool.back();
        e->prof_pool.pop_back();
      } else {
        GCA_CUDA(cudaEventCreate(&evs[i]));
      }
      e->prof_events.push_back(evs[i]);
    }
    ev = evs;
  }
  GCA_CUDA(launch_step(e->mode == GCA_MODE_FAITHFUL, e->draws == GCA_DRAWS_TAPE, a, (cudaStream_t)stream, ev));
  return GCA_OK;
}

int gca_step_launches(gca_env* e) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  return step_launch_count(e->draws == GCA_DRAWS_TAPE, e->s.N, e->cfg.obs_kind, e->cfg.intruder_turns && e->s.ihs);
}

int gca_check(gca_env* e) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(cudaDeviceSynchronize());
  int flag = 0;
  GCA_CUDA(cudaMemcpy(&flag, e->s.error_flag, sizeof(int), cudaMemcpyDeviceToHost));
  if (flag & 1) return fail(GCA_ERR_STATE, "a streaming lane timed out waiting for its ownship record (step_intruders_kernel)");
  return GCA_OK;
}

int gca_profile_enable(gca_env* e, int on) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  e->profiling = on != 0;
  return GCA_OK;
}

int gca_profile_read(gca_env* e, gca_step_profile* out) {
  if (!e || !out) return fail(GCA_ERR_INVALID, "env/out is NULL");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(cudaDeviceSynchronize());
  gca_step_profile p = {};
  for (size_t i = 0; i + 4 < e->prof_events.size(); i += 5) {
    float ms[4];
    for (int j = 0; j < 4; ++j) GCA_CUDA(cudaEventElapsedTime(&ms[j], e->prof_events[i + j], e->prof_events[i + j + 1]));
    p.steps += 1;
    p.own_ms += ms[0]; p.intruders_ms += ms[1]; p.finish_ms += ms[2]; p.spawn_ms += ms[3];
  }
  e->prof_pool.insert(e->prof_pool.end(), e->prof_events.begin(), e->prof_events.end());
  e->prof_events.clear();
  *out = p;
  return GCA_OK;
}

int gca_observe(gca_env* e, const gca_out* out, void* stream) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (int rc = check_out(e, out, false)) return rc;
  GCA_CUDA(cudaSetDevice(e->device));
  const StepArgs a = make_args(e, nullptr, nullptr, out, 0);
  GCA_CUDA(launch_observe(e->mode == GCA_MODE_FAITHFUL, a, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_read_counters(gca_env* e, int32_t* counters, void* stream) {
  if (!e || !counters) return fail(GCA_ERR_INVALID, "env/counters is NULL");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(cudaMemcpyAsync(counters, e->s.counters, (size_t)e->s.B * sizeof(int4), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return GCA_OK;
}

// ------------------------------------------------------------------------------ host-buffer path
static void release_host_path(gca_env* e) {
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  e->stream = e->copy_stream = nullptr;
  for (int i = 0; i < 2; ++i) {
    if (e->ev_step[i]) cudaEventDestroy(e->ev_step[i]);
    if (e->ev_copy[i]) cudaEventDestroy(e->ev_copy[i]);
    e->ev_step[i] = e->ev_copy[i] = nullptr;
  }
}

static int ensure_host_path(gca_env* e) {
  if (e->stream) return GCA_OK;
  if (e->draws != GCA_DRAWS_PHILOX) return fail(GCA_ERR_STATE, "the host-buffer path needs GCA_DRAWS_PHILOX");
  GCA_CUDA(cudaSetDevice(e->device));
  const size_t B = (size_t)e->s.B, rs = real_size(e);
  int rc = GCA_OK;
  uint8_t* p = nullptr;
  for (int k = 0; k < 2 && !rc; ++k) {
    if (!rc) { rc = dev_alloc(e, &p, B * 2 * sizeof(double)); e->d_actions[k] = p; }
    if (!rc) { rc = dev_alloc(e, &p, B * (size_t)e->D * rs); e->d_out[k].obs = p; }
    if (!rc) { rc = dev_alloc(e, &p, B * 2 * rs); e->d_out[k].achieved = p; }
    if (!rc) { rc = dev_alloc(e, &p, B * 2 * rs); e->d_out[k].desired = p; }
    if (!rc) { rc = dev_alloc(e, &p, B * rs); e->d_out[k].reward = p; }
    if (!rc) { rc = dev_alloc(e, &p, B); e->d_out[k].done = p; }
    if (!rc) { rc = dev_alloc(e, &p, B); e->d_out[k].info = p; }
    if (!rc && e->cfg.shaped_nearest) { rc = dev_alloc(e, &p, B * rs); e->d_out[k].nearest = p; }
  }
  if (rc) return rc;                                       // (the buffers stay in e->allocs; the path stays unset)
  cudaStream_t st = nullptr, cs = nullptr;
  cudaError_t ce = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
  for (int i = 0; i < 2 && ce == cudaSuccess; ++i) {
    ce = cudaEventCreateWithFlags(&e->ev_step[i], cudaEventDisableTiming);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&e->ev_copy[i], cudaEventDisableTiming);
  }
  e->stream = st;
  e->copy_stream = cs;
  if (ce != cudaSuccess) {
    release_host_path(e);
    return cuda_fail(ce, "creating the host path's streams / events");
  }
  return GCA_OK;
}

// downloads of one set of device-side outputs, enqueued on `st`
static int enqueue_copy_out(gca_env* e, const gca_out& d, const gca_out* h, bool with_reward, cudaStream_t st) {
  const size_t B = (size_t)e->s.B, rs = real_size(e);
  const bool her = e->cfg.obs_kind == GCA_OBS_HER || e->cfg.obs_kind == GCA_OBS_DHER || e->cfg.obs_kind == GCA_OBS_NEAREST;
  if (h->obs && e->D) GCA_CUDA(cudaMemcpyAsync(h->obs, d.obs, B * (size_t)e->D * rs, cudaMemcpyDeviceToHost, st));
  if (her && h->achieved) GCA_CUDA(cudaMemcpyAsync(h->achieved, d.achieved, B * 2 * rs, cudaMemcpyDeviceToHost, st));
  if (her && h->desired) GCA_CUDA(cudaMemcpyAsync(h->desired, d.desired, B * 2 * rs, cudaMemcpyDeviceToHost, st));
  if (with_reward && h->reward) GCA_CUDA(cudaMemcpyAsync(h->reward, d.reward, B * rs, cudaMemcpyDeviceToHost, st));
  if (h->done) GCA_CUDA(cudaMemcpyAsync(h->done, d.done, B, cudaMemcpyDeviceToHost, st));
  if (h->info) GCA_CUDA(cudaMemcpyAsync(h->info, d.info, B, cudaMemcpyDeviceToHost, st));
  if (h->nearest && d.nearest) GCA_CUDA(cudaMemcpyAsync(h->nearest, d.nearest, B * rs, cudaMemcpyDeviceToHost, st));
  return GCA_OK;
}

int gca_step_host_begin(gca_env* e, const void* actions_host, int auto_reset, const gca_out* host_out) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (!actions_host || !host_out) return fail(GCA_ERR_INVALID, "actions/out is NULL");
  if (int rc = ensure_host_path(e)) return rc;
  if (e->host_begun - e->host_waited >= 2) return fail(GCA_ERR_STATE, "two steps are already in flight: call gca_step_host_wait first");
  const int k = (int)(e->host_begun & 1ull);
  const size_t B = (size_t)e->s.B;
  const size_t abytes = e->cfg.action_kind == GCA_ACT_CONTINUOUS2 ? B * 2 * real_size(e) : B * sizeof(int32_t);
  GCA_CUDA(cudaMemcpyAsync(e->d_actions[k], actions_host, abytes, cudaMemcpyHostToDevice, e->stream));
  // buffer set k was last downloaded by the step begun two calls ago: its copy must have read it
  if (e->host_begun >= 2) GCA_CUDA(cudaStreamWaitEvent(e->stream, e->ev_copy[k], 0));
  if (int rc = gca_step(e, e->d_actions[k], nullptr, auto_reset, &e->d_out[k], e->stream)) return rc;
  GCA_CUDA(cudaEventRecord(e->ev_step[k], e->stream));
  GCA_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_step[k], 0));
  if (int rc = enqueue_copy_out(e, e->d_out[k], host_out, true, e->copy_stream)) return rc;
  GCA_CUDA(cudaEventRecord(e->ev_copy[k], e->copy_stream));
  e->host_begun += 1;
  return GCA_OK;
}

int gca_step_host_wait(gca_env* e) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (e->host_begun == e->host_waited) return fail(GCA_ERR_STATE, "no step in flight");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(cudaEventSynchronize(e->ev_copy[(int)(e->host_waited & 1ull)]));
  e->host_waited += 1;
  return GCA_OK;
}

int gca_step_host(gca_env* e, const void* actions_host, int auto_reset, const gca_out* host_out) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  while (e->host_begun != e->host_waited)                  // (steps begun asynchronously come first)
    if (int rc = gca_step_host_wait(e)) return rc;
  if (int rc = gca_step_host_begin(e, actions_host, auto_reset, host_out)) return rc;
  return gca_step_host_wait(e);
}

int gca_reset_host(gca_env* e, const gca_out* host_out) {
  if (!e) return fail(GCA_ERR_INVALID, "env is NULL");
  if (!host_out) return fail(GCA_ERR_INVALID, "out is NULL");
  if (int rc = ensure_host_path(e)) return rc;
  while (e->host_begun != e->host_waited)
    if (int rc = gca_step_host_wait(e)) return rc;
  GCA_CUDA(cudaStreamSynchronize(e->copy_stream));
  if (int rc = gca_reset(e, nullptr, nullptr, &e->d_out[0], e->stream)) return rc;
  if (int rc = enqueue_copy_out(e, e->d_out[0], host_out, false, e->stream)) return rc;
  GCA_CUDA(cudaStreamSynchronize(e->stream));
  return GCA_OK;
}

// ------------------------------------------------------------------------------ full-state access
int gca_get_state(gca_env* e, const gca_host_state* h) {
  if (!e || !h) return fail(GCA_ERR_INVALID, "env/state is NULL");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(cudaDeviceSynchronize());
  const DevState& s = e->s;
  const size_t B = (size_t)s.B, N = (size_t)s.N;
  if (h->own_pos) GCA_CUDA(cudaMemcpy(h->own_pos, s.own_pos, B * sizeof(float2), cudaMemcpyDeviceToHost));
  if (h->own_hs) GCA_CUDA(cudaMemcpy(h->own_hs, s.own_hs, B * sizeof(double2), cudaMemcpyDeviceToHost));
  if (h->own_vel) GCA_CUDA(cudaMemcpy(h->own_vel, s.own_vel, B * sizeof(double2), cudaMemcpyDeviceToHost));
  if (h->own_vel_is_f32) GCA_CUDA(cudaMemcpy(h->own_vel_is_f32, s.own_vel_f32, B, cudaMemcpyDeviceToHost));
  if (h->goal) GCA_CUDA(cudaMemcpy(h->goal, s.goal, B * sizeof(double2), cudaMemcpyDeviceToHost));
  if (h->no_conflict || h->ep_steps || h->tick) {
    std::vector<int4> c(B);
    GCA_CUDA(cudaMemcpy(c.data(), s.counters, B * sizeof(int4), cudaMemcpyDeviceToHost));
    for (size_t b = 0; b < B; ++b) {
      if (h->no_conflict) h->no_conflict[b] = c[b].x;
      if (h->ep_steps) h->ep_steps[b] = c[b].y;
      if (h->tick) h->tick[b] = (uint32_t)c[b].z;
    }
  }
  if (N == 0 || !(h->ipos || h->ivel || h->iflag || h->ipos_is_f64 || h->ihs)) return GCA_OK;
  const bool faith = e->mode == GCA_MODE_FAITHFUL;
  HostPlanes hp;
  if (int rc = hp.download(s, faith)) return rc;
  for (size_t b = 0; b < B; ++b) {
    for (size_t i = 0; i < N; ++i) {
      const size_t k = b * N + i;
      if (h->ipos) {
        if (faith) {
          const double2 p = *reinterpret_cast<const double2*>(hp.plane_of(s, b) + ipos_offset(s, true, b, (int)i));
          h->ipos[2 * k] = p.x; h->ipos[2 * k + 1] = p.y;
        } else {
          const float2 p = *reinterpret_cast<const float2*>(hp.plane_of(s, b) + ipos_offset(s, false, b, (int)i));
          h->ipos[2 * k] = (double)p.x; h->ipos[2 * k + 1] = (double)p.y;
        }
      }
      if (h->ivel) {
        const float2 v = *reinterpret_cast<const float2*>(hp.vel.data() + ivel_offset(s, b, (int)i));
        h->ivel[2 * k] = v.x; h->ivel[2 * k + 1] = v.y;
      }
      const size_t fi = flag_index(s, b, (int)(i / 32));
      if (h->iflag) h->iflag[k] = (hp.cf[fi] >> (i % 32)) & 1u;
      if (h->ipos_is_f64) h->ipos_is_f64[k] = faith ? ((hp.df[fi] >> (i % 32)) & 1u) : 0;
      if (h->ihs) {
        const double2 v = s.ihs ? hp.hs[ihs_index(s, b, (int)i)] : make_double2(0.0, 0.0);
        h->ihs[2 * k] = v.x; h->ihs[2 * k + 1] = v.y;
      }
    }
  }
  return GCA_OK;
}

int gca_set_state(gca_env* e, const gca_host_state* h) {
  if (!e || !h) return fail(GCA_ERR_INVALID, "env/state is NULL");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(cudaDeviceSynchronize());
  const DevState& s = e->s;
  const size_t B = (size_t)s.B, N = (size_t)s.N;
  if (h->own_pos) GCA_CUDA(cudaMemcpy(s.own_pos, h->own_pos, B * sizeof(float2), cudaMemcpyHostToDevice));
  if (h->own_hs) GCA_CUDA(cudaMemcpy(s.own_hs, h->own_hs, B * sizeof(double2), cudaMemcpyHostToDevice));
  if (h->own_vel) GCA_CUDA(cudaMemcpy(s.own_vel, h->own_vel, B * sizeof(double2), cudaMemcpyHostToDevice));
  if (h->own_vel_is_f32) GCA_CUDA(cudaMemcpy(s.own_vel_f32, h->own_vel_is_f32, B, cudaMemcpyHostToDevice));
  if (h->goal) GCA_CUDA(cudaMemcpy(s.goal, h->goal, B * sizeof(double2), cudaMemcpyHostToDevice));
  const bool faith = e->mode == GCA_MODE_FAITHFUL;
  HostPlanes hp;
  if (int rc = hp.download(s, faith)) return rc;                      // keep what the view omits
  for (size_t b = 0; b < B; ++b) {
    const int old_plane = hp.cnt[b].z & 1;
    if (h->no_conflict) hp.cnt[b].x = h->no_conflict[b];
    if (h->ep_steps) hp.cnt[b].y = h->ep_steps[b];
    if (h->tick) hp.cnt[b].z = (int)h->tick[b];
    const int new_plane = hp.cnt[b].z & 1;                            // the tick selects the current position plane
    const uint8_t* from = hp.pos.data() + (size_t)old_plane * s.pos_plane;
    uint8_t* to = hp.pos.data() + (size_t)new_plane * s.pos_plane;
    for (int w = 0; w < s.W; ++w) {
      if (h->iflag) hp.cf[flag_index(s, b, w)] = 0u;
      if (h->ipos_is_f64 && faith) hp.df[flag_index(s, b, w)] = 0u;
    }
    for (size_t i = 0; i < N; ++i) {
      const size_t k = b * N + i;
      const size_t po = ipos_offset(s, faith, b, (int)i);
      if (faith) {
        *reinterpret_cast<double2*>(to + po) = h->ipos ? make_double2(h->ipos[2 * k], h->ipos[2 * k + 1])
                                                       : *reinterpret_cast<const double2*>(from + po);
      } else {
        // FAST positions are stored as non-negative-zero f32 (the map test of the streaming pass compares bit
        // patterns); -0.0 and +0.0 are the same position for every rule of the reference.
        *reinterpret_cast<float2*>(to + po) = h->ipos ? make_float2((float)h->ipos[2 * k] + 0.0f, (float)h->ipos[2 * k + 1] + 0.0f)
                                                      : *reinterpret_cast<const float2*>(from + po);
      }
      if (h->ivel)
        *reinterpret_cast<float2*>(hp.vel.data() + ivel_offset(s, b, (int)i)) = make_float2(h->ivel[2 * k], h->ivel[2 * k + 1]);
      const size_t fi = flag_index(s, b, (int)(i / 32));
      if (h->iflag && h->iflag[k]) hp.cf[fi] |= 1u << (i % 32);
      if (h->ipos_is_f64 && faith && h->ipos_is_f64[k]) hp.df[fi] |= 1u << (i % 32);
      if (h->ihs && s.ihs) hp.hs[ihs_index(s, b, (int)i)] = make_double2(h->ihs[2 * k], h->ihs[2 * k + 1]);
    }
  }
  return hp.upload(s, faith);
}

int gca_compute_reward(const void* ag, const void* g, int64_t m, double radius, int kind, int is_f64, float* out,
                       int device, void* stream) {
  if (m < 0 || (m > 0 && (!ag || !g || !out))) return fail(GCA_ERR_INVALID, "bad buffers");
  if (kind != GCA_OBS_HER && kind != GCA_OBS_DHER) return fail(GCA_ERR_INVALID, "kind must be GCA_OBS_HER or GCA_OBS_DHER");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_compute_reward(ag, (long long)m, g, (long long)m, radius, kind, is_f64, out, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_compute_reward_tiled(const void* ag, int64_t n_ag, const void* g, int64_t m, double radius, int kind, int is_f64,
                             float* out, int device, void* stream) {
  if (m < 0 || n_ag <= 0 || (m > 0 && (!ag || !g || !out)) || m % n_ag) return fail(GCA_ERR_INVALID, "bad buffers (m must be a multiple of n_ag)");
  if (kind != GCA_OBS_HER && kind != GCA_OBS_DHER) return fail(GCA_ERR_INVALID, "kind must be GCA_OBS_HER or GCA_OBS_DHER");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_compute_reward(ag, (long long)n_ag, g, (long long)m, radius, kind, is_f64, out, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_input_reward(const void* rows, int64_t m, int dim, int is_f64, const gca_input_reward_cfg* cfg, double* out,
                     uint8_t* done, int device, void* stream) {
  if (m < 0 || !cfg || (m > 0 && (!rows || !out))) return fail(GCA_ERR_INVALID, "bad buffers");
  if (dim < 4 || (cfg->has_intruders && cfg->n_listed > 0 && (cfg->n_listed - 1) * 4 + 5 >= dim))
    return fail(GCA_ERR_INVALID, "rows are shorter than the entries compute_input_reward reads");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_input_reward(rows, (long long)m, dim, is_f64, cfg, out, done, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_monitor_update(const void* reward, int is_f64, const uint8_t* done, int64_t n_envs, float* ep_return,
                       int32_t* ep_length, gca_episode_record* ring, int64_t ring_capacity,
                       unsigned long long* ring_count, uint32_t step, int device, void* stream) {
  if (n_envs < 0 || ring_capacity <= 0 || (n_envs > 0 && (!reward || !done || !ep_return || !ep_length || !ring || !ring_count)))
    return fail(GCA_ERR_INVALID, "bad arguments");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_monitor_update(reward, is_f64, done, (long long)n_envs, ep_return, ep_length, ring,
                                 (long long)ring_capacity, ring_count, step, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_stats_update(const uint8_t* done, const uint8_t* info, int64_t n_envs, unsigned long long* stats, int device,
                     void* stream) {
  if (n_envs < 0 || (n_envs > 0 && (!done || !info || !stats))) return fail(GCA_ERR_INVALID, "bad arguments");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_stats_update(done, info, (long long)n_envs, stats, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_her_sample(const gca_her_episodes* ep, int64_t n_episodes, int T, int dim_o, int dim_u, int dim_g, int is_f64,
                   int64_t batch, double future_p, double goal_radius, int reward_kind, const gca_her_draws* draws,
                   uint64_t seed, uint32_t call, const gca_her_transitions* out, int device, void* stream) {
  if (!ep || !out || n_episodes <= 0 || T <= 0 || dim_o <= 0 || dim_u <= 0 || batch < 0)
    return fail(GCA_ERR_INVALID, "bad arguments");
  if (dim_g != 2) return fail(GCA_ERR_INVALID, "goals are 2-D (achieved_goal / desired_goal of the GoalEnv variants)");
  if (reward_kind != GCA_OBS_HER && reward_kind != GCA_OBS_DHER) return fail(GCA_ERR_INVALID, "reward_kind must be GCA_OBS_HER or GCA_OBS_DHER");
  if (!ep->o || !ep->u || !ep->g || !ep->ag) return fail(GCA_ERR_INVALID, "episode arrays are NULL");
  if (batch > 0 && (!out->o || !out->u || !out->g || !out->ag || !out->o_2 || !out->ag_2 || !out->r))
    return fail(GCA_ERR_INVALID, "transition arrays are NULL");
  if (draws && (!draws->episode_idxs || !draws->t_samples || !draws->u_her || !draws->u_offset))
    return fail(GCA_ERR_INVALID, "draws need all four arrays");
  if (!(future_p >= 0.0 && future_p <= 1.0)) return fail(GCA_ERR_INVALID, "future_p must be in [0, 1]");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_her_sample(ep, (long long)n_episodes, T, dim_o, dim_u, dim_g, is_f64, (long long)batch, future_p,
                             goal_radius, reward_kind, draws, seed, call, out, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_raster(gca_env* e, const uint8_t* sprites, uint8_t* frames, int64_t env_stride, int64_t plane_stride,
               int n_planes, int slot, const uint8_t* clear_mask, void* stream) {
  if (!e || !sprites || !frames) return fail(GCA_ERR_INVALID, "env/sprites/frames is NULL");
  if (e->s.N > GCA_RASTER_MAX_INTRUDERS) return fail(GCA_ERR_STATE, "the rasteriser supports at most 126 intruders");
  const int W = (int)e->cfg.window_width, H = (int)e->cfg.window_height;
  if (W != e->cfg.window_width || H != e->cfg.window_height || W % 16 || H % 4 || W <= 0 || H <= 0)
    return fail(GCA_ERR_STATE, "the rasteriser needs an integer window with width % 16 == 0 and height % 4 == 0");
  if (n_planes < 1 || slot < 0 || slot >= n_planes) return fail(GCA_ERR_INVALID, "bad plane selection");
  if (plane_stride % 4 || env_stride % 4) return fail(GCA_ERR_INVALID, "strides must be multiples of 4 bytes");
  // the kernel reads sprites and writes frames 4 bytes at a time: with the stride rule above, 4-byte aligned
  // pointers make every such access aligned
  if (reinterpret_cast<uintptr_t>(frames) % 4) return fail(GCA_ERR_INVALID, "frames must be 4-byte aligned");
  if (reinterpret_cast<uintptr_t>(sprites) % 4) return fail(GCA_ERR_INVALID, "sprites must be 4-byte aligned");
  if (raster_smem_bytes(W / 4, H / 4) > kRasterSmemMax || W / 4 > 32767 || H / 4 > 32767)
    return fail(GCA_ERR_STATE, "the rasteriser keeps the whole " + std::to_string(W / 4) + "x" + std::to_string(H / 4) +
                                   " output plane of the " + std::to_string(W) + "x" + std::to_string(H) +
                                   " canvas in shared memory: " + std::to_string(raster_smem_bytes(W / 4, H / 4)) +
                                   " bytes, more than the " + std::to_string(kRasterSmemMax) + " a block may use");
  GCA_CUDA(cudaSetDevice(e->device));
  GCA_CUDA(launch_raster(e->s, e->mode == GCA_MODE_FAITHFUL, W, H, sprites, frames, (long long)env_stride,
                         (long long)plane_stride, n_planes, slot, clear_mask, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_mcts_move(const gca_mcts_config* cfg, int n_intruders, double* states, const int32_t* actions, uint8_t* flags,
                  int64_t m, const gca_tape* tape, uint64_t seed, uint32_t id0, int first_frame, int device,
                  void* stream) {
  if (!cfg || n_intruders < 0 || m < 0 || (m > 0 && (!states || !actions || !flags))) return fail(GCA_ERR_INVALID, "bad arguments");
  if (tape && (!tape->values || !tape->cursor)) return fail(GCA_ERR_INVALID, "tape needs values and cursor");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_mcts_move(cfg, n_intruders, states, actions, flags, (long long)m, tape ? tape->values : nullptr,
                            tape ? (long long)tape->stride : 0, tape ? reinterpret_cast<long long*>(tape->cursor) : nullptr,
                            seed, id0, first_frame, (cudaStream_t)stream));
  return GCA_OK;
}

int gca_mcts_playouts(const gca_mcts_config* cfg, int n_intruders, const double* roots, int64_t n_roots, int playouts,
                      int depth, const int8_t* first_action, uint64_t seed, uint32_t root_id0, double* rewards,
                      int8_t* first_out, uint8_t* flags, int device, void* stream) {
  if (!cfg || n_intruders < 0 || n_roots < 0 || playouts <= 0 || depth < 0 || (n_roots > 0 && (!roots || !rewards)))
    return fail(GCA_ERR_INVALID, "bad arguments");
  if (cfg->simulate_frame <= 0) return fail(GCA_ERR_INVALID, "simulate_frame must be positive");
  if (cfg->random_intruders && (size_t)n_intruders * 52 * 4 > 200 * 1024)
    return fail(GCA_ERR_INVALID, "random_intruders playouts keep 4 x 52 N bytes in shared memory: at most 984 intruders");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_mcts_playouts(cfg, n_intruders, roots, (long long)n_roots, playouts, depth, first_action, seed,
                                root_id0, rewards, first_out, flags, (cudaStream_t)stream));
  return GCA_OK;
}

int64_t gca_mcts_search_workspace(const gca_mcts_config* cfg, int n_intruders, int64_t n_roots, int simulations,
                                  int depth) {
  if (!cfg || n_intruders < 0 || n_roots < 0 || simulations < 0 || depth < 0) return -1;
  return (int64_t)mcts_search_workspace_bytes(cfg, n_intruders, (long long)n_roots, simulations, depth);
}

int gca_mcts_search(const gca_mcts_config* cfg, int n_intruders, const double* roots, int64_t n_roots, int simulations,
                    int depth, uint64_t seed, uint32_t root_id0, void* workspace, int64_t workspace_bytes,
                    int32_t* best_action, double* child_n, double* child_q, int32_t* child_action, int device,
                    void* stream) {
  if (!cfg || n_intruders < 0 || n_roots < 0 || simulations < 0 || depth < 0 || (n_roots > 0 && (!roots || !best_action)))
    return fail(GCA_ERR_INVALID, "bad arguments");
  if (cfg->simulate_frame <= 0) return fail(GCA_ERR_INVALID, "simulate_frame must be positive");
  if (cfg->position_sigma != 0.0 || cfg->random_intruders)
    return fail(GCA_ERR_STATE, "the device-resident search needs position_sigma == 0 and no random_intruders (use the node classes otherwise)");
  if (simulations > 32000 || depth > 127) return fail(GCA_ERR_INVALID, "at most 32000 simulations and depth 127");
  const int64_t need = gca_mcts_search_workspace(cfg, n_intruders, n_roots, simulations, depth);
  if (n_roots > 0 && (!workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(workspace) % 16))
    return fail(GCA_ERR_INVALID, "workspace missing, misaligned or smaller than gca_mcts_search_workspace()");
  GCA_CUDA(cudaSetDevice(device));
  GCA_CUDA(launch_mcts_search(cfg, n_intruders, roots, (long long)n_roots, simulations, depth, seed, root_id0, workspace,
                              best_action, child_n, child_q, child_action, (cudaStream_t)stream));
  return GCA_OK;
}

}  // extern "C"
