// mgym_api.cu -- C ABI (include/mgym.h) over the CUDA kernels.  No torch types, no CPU fallback.
#include <dlfcn.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <string>

#include "../../include/mgym.h"
#include "mgym_kernels.cuh"

// NCCL is resolved at run time (dlsym), so the library has no link dependency on it; the two enum values
// mgym_stats_allreduce passes are taken from <nccl.h> where the header is installed and checked against the
// values the header-less build assumes (NCCL has kept them since 2.0).
#if defined(__has_include)
#if __has_include(<nccl.h>)
#include <nccl.h>
#define MGYM_HAVE_NCCL_H 1
#endif
#endif
namespace {
#ifdef MGYM_HAVE_NCCL_H
constexpr int kNcclFloat64 = (int)ncclFloat64, kNcclSum = (int)ncclSum;
static_assert(kNcclFloat64 == 8 && kNcclSum == 0, "NCCL enum values changed: update the header-less fallback below");
#else
constexpr int kNcclFloat64 = 8, kNcclSum = 0;  // ncclFloat64, ncclSum (nccl.h 2.x)
#endif
}  // namespace

using namespace mgym;

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct mgym_env {
  int kind = 0;
  uint64_t n = 0;
  int device = 0;
  uint64_t seed = 0;
  mgym_config cfg{};
  int cnt_mode = CNT_U32;
  bool vec4 = false;  // n % 4 == 0 and env_index_base % 4 == 0

  float* state = nullptr;
  void* steps = nullptr;
  uint32_t* sbt = nullptr;
  float* ep_return = nullptr;
  float* reset_pool = nullptr;
  uint64_t pool_len = 0;
  unsigned long long* stats = nullptr;  // 5 x 8 bytes
  uint32_t* bad_action = nullptr;
  float* params = nullptr;  // per-env physics parameters [P][n] (mgym_set_params), null = the kind's constants
  // per-episode redraw ranges (mgym_set_param_redraw): every reset draws the env's parameters from U[lo, hi)
  bool redraw = false;
  float redraw_lo[MAX_PARAMS] = {}, redraw_hi[MAX_PARAMS] = {};

  uint64_t t = 0;         // steps executed since creation
  uint64_t n_resets = 0;  // explicit reset calls since creation
  EnvConsts k{};
  int num_sms = 0;

  // device staging for mgym_step_host
  void* h_actions = nullptr;
  float* h_obs = nullptr;
  float* h_reward = nullptr;
  uint8_t* h_flags = nullptr;
  unsigned long long* work = nullptr;   // ticket counters: step on the caller's stream, pipe streams 0 and 1, rollout
  uint64_t work_issued[3] = {0, 0, 0};  // tickets handed to launches so far, per counter
  int work_slot = 0;                    // counter the next TMA launch uses
  // device clock (cfg.device_clock): {step index, first ticket of the step counter, finished CTAs of the
  // running launch}; see KernelParams::t_dev / adv_clock
  unsigned long long* clock = nullptr;
  uint64_t call_tickets = 0;            // tickets the TMA launches of the running call draw from counter 0
  cudaStream_t pipe_stream[2] = {nullptr, nullptr};
  cudaEvent_t pipe_event[3] = {nullptr, nullptr, nullptr};
};

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define MGYM_CUDA(expr)                                                                            \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(e_ == cudaErrorMemoryAllocation ? MGYM_ERR_OUT_OF_MEMORY : MGYM_ERR_CUDA,        \
                  "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__);    \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

constexpr int kStateDim[MGYM_NUM_KINDS] = {4, 2, 2, 2, 4};
constexpr int kObsDim[MGYM_NUM_KINDS] = {4, 2, 2, 3, 6};
constexpr int kContinuous[MGYM_NUM_KINDS] = {0, 0, 1, 1, 0};
constexpr int kNumActions[MGYM_NUM_KINDS] = {2, 3, 0, 0, 3};
const char* const kNames[MGYM_NUM_KINDS] = {"CartPole-v1", "MountainCar-v0", "MountainCarContinuous-v0",
                                            "Pendulum-v1", "Acrobot-v1"};

// Per-env physics parameters (mgym_set_params): count, names, defaults (the constants of make_consts and of the
// device code) and the ones that must be > 0 (bit c = parameter c).  Acrobot has none.
constexpr int kNumParams[MGYM_NUM_KINDS] = {6, 2, 2, 3, 0};
const char* const kParamNames[MGYM_NUM_KINDS][6] = {
    {"gravity", "masscart", "masspole", "length", "force_mag", "tau"},
    {"force", "gravity"},
    {"power", "gravity"},
    {"g", "m", "l"},
    {}};
constexpr float kParamDefaults[MGYM_NUM_KINDS][6] = {
    {9.8f, 1.0f, 0.1f, 0.5f, 10.0f, 0.02f}, {0.001f, 0.0025f}, {0.0015f, 0.0025f}, {10.0f, 1.0f, 1.0f}, {}};
constexpr uint32_t kParamPositive[MGYM_NUM_KINDS] = {0x2Eu, 0u, 0u, 0x6u, 0u};
static_assert(Env<0>::NP == 6 && Env<1>::NP == 2 && Env<2>::NP == 2 && Env<3>::NP == 3 && Env<4>::NP == 0,
              "parameter tables and Env<KIND>::NP disagree");

bool valid_kind(int kind) { return kind >= 0 && kind < MGYM_NUM_KINDS; }
size_t counter_width(int cnt_mode) { return cnt_mode == CNT_S16 ? 2 : 4; }
size_t action_size(int kind) { return kContinuous[kind] ? sizeof(float) : sizeof(uint8_t); }
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// f32 constants, evaluated in the constructors' operator order (cartpole.rs:45-56,
// mountain_car.rs:35-40).  volatile keeps the host compiler from re-associating.
EnvConsts make_consts(int kind, const mgym_config& cfg) {
  EnvConsts k{};
  volatile float masscart = 1.0f, masspole = 0.1f, length = 0.5f, tau = 0.02f;
  k.gravity = 9.8f;
  k.masspole = masspole;
  k.total_mass = masspole + masscart;
  k.rcp_total_mass = (float)(1.0 / (double)k.total_mass);  // RN(1/total_mass), see fdiv_const_fast
  k.length = length;
  k.polemass_length = masspole * length;
  k.force_mag = 10.0f;
  k.tau = tau;
  volatile float half_tau = 0.5f * tau;
  k.half_tau = half_tau;
  k.half_tau_tau = half_tau * tau;
  volatile float th = 12.0f * 2.0f;
  th = th * 3.14159274101257324f;  // std::f32::consts::PI
  th = th / 360.0f;
  k.theta_threshold = th;
  k.x_threshold = 2.4f;
  volatile float four = 4.0f, three = 3.0f;
  k.four_thirds = four / three;

  k.min_position = -1.2f;
  k.max_position = 0.6f;
  k.max_speed = 0.07f;
  k.goal_position = 0.5f;
  k.goal_velocity = cfg.goal_velocity;
  k.force = 0.001f;
  k.mc_gravity = 0.0025f;
  k.power = 0.0015f;

  volatile float m1 = 1.0f, m2 = 1.0f, l1 = 1.0f, lc1 = 0.5f, lc2 = 0.5f, g = 9.8f, dt = 0.2f;
  volatile float a = m1 * lc1, b = m2 * l1;
  volatile float ab = a + b;
  k.m1lc1g = ab * g;
  volatile float c = m2 * lc2;
  k.m2lc2g = c * g;
  k.dt = dt;
  k.dt2 = dt / 2.0f;
  k.dt6 = dt / 6.0f;
  volatile float pi = PI_F;
  k.max_vel_1 = 4.0f * pi;
  k.max_vel_2 = 9.0f * pi;

  k.one = 1.0f;
  k.r_alive = cfg.sutton_barto_reward ? 0.0f : 1.0f;   // cartpole.rs:311
  k.r_fell = cfg.sutton_barto_reward ? -1.0f : 1.0f;   // cartpole.rs:322
  k.r_after = cfg.sutton_barto_reward ? -1.0f : 0.0f;  // cartpole.rs:338
  k.is_euler = cfg.is_euler;
  k.sutton_barto = cfg.sutton_barto_reward;
  k.max_steps = (kind == MGYM_CARTPOLE_V1) ? 0 : cfg.max_episode_steps;
  return k;
}

KernelParams base_params(const mgym_env* e) {
  KernelParams p{};
  p.state = e->state;
  p.steps = e->steps;
  p.sbt = e->sbt;
  p.ep_return = e->ep_return;
  p.reset_pool = e->pool_len ? e->reset_pool : nullptr;
  p.pool_len = e->pool_len;
  p.stats = (e->cfg.auto_reset && e->cfg.track_stats) ? e->stats : nullptr;
  p.n = e->n;
  p.first = 0;
  p.ld = e->n;
  p.seed = e->seed;
  p.keys = philox_keys(e->seed);
  p.t_dev = e->cfg.device_clock ? e->clock : nullptr;
  p.base_dev = nullptr;  // set by launch_step_tma for counter 0
  p.env_base = e->cfg.env_index_base;
  p.t = e->t;
  p.k = e->k;
  return p;
}

// Occupancy of a kernel is a per-device constant: query it once per (kernel instantiation, device).
constexpr int kMaxDevices = 64;

// Every step_kernel / rollout_kernel instantiation has the same function-pointer TYPE, so the table is keyed by
// the kernel's address (and the device), not by a template parameter.
struct OccupancyCache {
  static constexpr int kSlots = 256;
  std::mutex mu;
  const void* key[kSlots] = {};
  int dev[kSlots] = {};
  int per_sm[kSlots] = {};
  int used = 0;
  int find(const void* k, int d) {
    std::lock_guard<std::mutex> lock(mu);
    for (int i = 0; i < used; ++i)
      if (key[i] == k && dev[i] == d) return per_sm[i];
    return 0;
  }
  void put(const void* k, int d, int v) {
    std::lock_guard<std::mutex> lock(mu);
    if (used < kSlots) key[used] = k, dev[used] = d, per_sm[used] = v, ++used;
  }
};
OccupancyCache g_occupancy;

template <typename KP>
int launch_persistent(void (*kernel)(KP), const mgym_env* e, const KP& p, uint64_t groups, cudaStream_t st) {
  constexpr int threads = 256;
  int per_sm = g_occupancy.find(reinterpret_cast<const void*>(kernel), e->device);
  if (per_sm == 0) {
    MGYM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0));
    if (per_sm < 1) per_sm = 1;
    g_occupancy.put(reinterpret_cast<const void*>(kernel), e->device, per_sm);
  }
  uint64_t blocks = (uint64_t)e->num_sms * per_sm;
  const uint64_t need = (groups + threads - 1) / threads;
  if (blocks > need) blocks = need;
  if (blocks < 1) blocks = 1;
  kernel<<<(unsigned)blocks, threads, 0, st>>>(p);
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

// TMA-staged step kernel (auto-reset, vector path, N a multiple of the 128-env warp tile)
template <int KIND, int CNT, bool AUTO = true, bool PARAMS = false, bool REDRAW = false>
int launch_step_tma(const mgym_env* ce, const KParams<PARAMS, REDRAW>& p_in, cudaStream_t st) {
  mgym_env* e = const_cast<mgym_env*>(ce);  // ticket accounting
  KParams<PARAMS, REDRAW> p = p_in;
  using L = TmaLayout<KIND, CNT, AUTO, PARAMS>;
  auto kernel = step_kernel_tma<KIND, CNT, AUTO, PARAMS, REDRAW>;
  constexpr int threads = TMA_THREADS;
  // the opt-in to > 48 KB of dynamic shared memory and the occupancy are per device
  static int cached_per_sm[kMaxDevices] = {};
  int per_sm = e->device < kMaxDevices ? cached_per_sm[e->device] : 0;
  if (per_sm == 0) {
    MGYM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::SMEM_BYTES));
    MGYM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, L::SMEM_BYTES));
    if (per_sm < 1) per_sm = 1;
    if (e->device < kMaxDevices) cached_per_sm[e->device] = per_sm;
  }
  // persistent CTAs, tiles handed out by tickets (see the producer warp)
  const uint64_t slots = (uint64_t)e->num_sms * per_sm;
  const uint64_t tiles = p.n / TMA_TILE;
  uint64_t blocks = tiles < slots ? tiles : slots;
  if (blocks < 1) blocks = 1;
  p.work_counter = e->work + e->work_slot;
  if (p.t_dev && e->work_slot == 0) {
    // device clock: the first ticket is read from clock[1], which moves on by this launch's tickets when the
    // launch ends (fused) or when clock_advance_kernel runs after the call.  One TMA launch per call draws
    // from counter 0 (the head of a ragged size, see dispatch_mode).
    p.base_dev = e->clock + 1;
    if (p.adv_clock)
      p.adv_tickets = tiles + blocks;
    else
      e->call_tickets += tiles + blocks;
  } else {
    p.work_base = e->work_issued[e->work_slot];
    e->work_issued[e->work_slot] += tiles + blocks;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)blocks);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = L::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MGYM_CUDA(cudaLaunchKernelEx(&cfg, kernel, p));
  return MGYM_OK;
}

// kind x vector width x auto/manual x counter representation (x per-env parameters (x per-episode redraw: auto-reset
// handles only, the host never asks for a manual form of it)) (x final observations: auto-reset rollouts only,
// mgym_rollout_final refuses manual handles before it gets here)
template <int KIND, int V, bool ROLLOUT, bool PARAMS = false, bool REDRAW = false, bool FINAL = false>
int dispatch_mode(const mgym_env* e, const KParams<PARAMS, REDRAW>& p, cudaStream_t st) {
  static_assert(!FINAL || ROLLOUT, "final observations are a rollout form");
  const uint64_t groups = p.n / V;
  const bool autor = e->cfg.auto_reset != 0;
  if constexpr (!ROLLOUT && V == 4) {
    // manual mode (the reference's protocol): counters are 32-bit, CartPole adds steps_beyond_terminated
    if constexpr (!REDRAW) {
      if (!autor && p.n % TMA_TILE == 0) return launch_step_tma<KIND, CNT_U32, false, PARAMS>(e, p, st);
    }
    if (autor && p.n % TMA_TILE == 0) {
      if constexpr (KIND == 0) {  // CartPole's handles are all CNT_S16 (500-step truncation, cartpole.rs:297)
        return launch_step_tma<KIND, CNT_S16, true, PARAMS, REDRAW>(e, p, st);
      } else {
        switch (e->cnt_mode) {
          case CNT_S16: return launch_step_tma<KIND, CNT_S16, true, PARAMS, REDRAW>(e, p, st);
          case CNT_S32_LAZY: return launch_step_tma<KIND, CNT_S32_LAZY, true, PARAMS, REDRAW>(e, p, st);
          default: return launch_step_tma<KIND, CNT_S32, true, PARAMS, REDRAW>(e, p, st);
        }
      }
    }
    if (p.n > TMA_TILE) {
      // ragged size: whole 1024-env tiles on the TMA kernel, the remaining (< 1024) envs on the vector kernel
      KParams<PARAMS, REDRAW> head = p, tail = p;
      head.adv_dt = 0;  // device clock: the tail launch (last of the call) moves the step index on
      head.n = p.n - p.n % TMA_TILE;
      tail.first = p.first + head.n;
      tail.n = p.n - head.n;
      int rc = dispatch_mode<KIND, 4, false, PARAMS, REDRAW>(e, head, st);
      if (rc != MGYM_OK) return rc;
      return dispatch_mode<KIND, 4, false, PARAMS, REDRAW>(e, tail, st);
    }
  }
  // rollout_kernel's FULL form: complete warp tiles and all three trajectory outputs
  [[maybe_unused]] const bool full = ROLLOUT && V == 4 && autor && p.n % (32 * V) == 0 && p.obs_out && p.reward_out &&
                                     p.flags_out;
#define MGYM_LAUNCH(AUTO_, CNT_)                                                                         \
  do {                                                                                                   \
    if constexpr (ROLLOUT) {                                                                             \
      if constexpr (AUTO_ && V == 4) {                                                                   \
        if (full)                                                                                        \
          return launch_persistent(rollout_kernel<KIND, V, AUTO_, CNT_, true, PARAMS, REDRAW, FINAL>, e, p, groups, st); \
      }                                                                                                  \
      return launch_persistent(rollout_kernel<KIND, V, AUTO_, CNT_, false, PARAMS, REDRAW, FINAL>, e, p, groups, st); \
    } else {                                                                                             \
      return launch_persistent(step_kernel<KIND, V, AUTO_, CNT_, PARAMS, REDRAW>, e, p, groups, st);     \
    }                                                                                                    \
  } while (0)
  if constexpr (!REDRAW && !FINAL) {
    if (!autor) MGYM_LAUNCH(false, CNT_U32);
  }
  if constexpr (KIND == 0) {
    MGYM_LAUNCH(true, CNT_S16);
  } else {
    switch (e->cnt_mode) {  // these kernels hold the count in registers: a lazy stamp is an ordinary one here
      case CNT_S16: MGYM_LAUNCH(true, CNT_S16);
      default: MGYM_LAUNCH(true, CNT_S32);
    }
  }
#undef MGYM_LAUNCH
}

// The handle's redraw ranges as the f64 box the kernels map Philox words into (the mapping of mgym_sample_params)
ParamBox redraw_box(const mgym_env* e) {
  ParamBox box{};
  for (int c = 0; c < MAX_PARAMS; ++c) {
    box.lo[c] = (double)e->redraw_lo[c];
    box.range[c] = (double)e->redraw_hi[c] - (double)e->redraw_lo[c];
  }
  return box;
}

// A handle with per-env parameters runs the PARAMS instantiations (kinds that have parameters only), an auto-reset
// one with redraw ranges the PARAMS + REDRAW instantiations (manual-mode steps never reset).
template <int KIND, bool ROLLOUT, bool FINAL>
int dispatch_kind(const mgym_env* e, const KernelParams& p, bool vec4, cudaStream_t st) {
  if constexpr (Env<KIND>::NP > 0) {
    if (e->params) {
      KernelParamsP pp;
      static_cast<KernelParams&>(pp) = p;
      pp.params = e->params;
      if (e->redraw && e->cfg.auto_reset) {
        KernelParamsR pr;
        static_cast<KernelParamsP&>(pr) = pp;
        pr.redraw = redraw_box(e);
        return vec4 ? dispatch_mode<KIND, 4, ROLLOUT, true, true, FINAL>(e, pr, st)
                    : dispatch_mode<KIND, 1, ROLLOUT, true, true, FINAL>(e, pr, st);
      }
      return vec4 ? dispatch_mode<KIND, 4, ROLLOUT, true, false, FINAL>(e, pp, st)
                  : dispatch_mode<KIND, 1, ROLLOUT, true, false, FINAL>(e, pp, st);
    }
  }
  return vec4 ? dispatch_mode<KIND, 4, ROLLOUT, false, false, FINAL>(e, p, st)
              : dispatch_mode<KIND, 1, ROLLOUT, false, false, FINAL>(e, p, st);
}

// FINAL: the rollout forms that also store final observations (mgym_rollout_final)
template <bool ROLLOUT, bool FINAL = false>
int dispatch(const mgym_env* e, const KernelParams& p, bool vec4, cudaStream_t st) {
#define MGYM_KIND(K_)                                               \
  case K_:                                                          \
    return dispatch_kind<K_, ROLLOUT, FINAL>(e, p, vec4, st)
  switch (e->kind) {
    MGYM_KIND(0);
    MGYM_KIND(1);
    MGYM_KIND(2);
    MGYM_KIND(3);
    MGYM_KIND(4);
  }
#undef MGYM_KIND
  return fail(MGYM_ERR_BAD_ARGUMENT, "bad kind %d", e->kind);
}

template <int KIND>
int launch_reset_kind(const mgym_env* e, const KernelParams& p, const uint8_t* mask, cudaStream_t st) {
  const bool sparse = mask && !p.obs_out && p.first == 0 && p.n % 16 == 0 && aligned16(mask);
  const unsigned blocks = sparse ? (unsigned)((p.n / 16 + 255) / 256) : (unsigned)((p.n + 255) / 256);
#define MGYM_RESET(CNT_)                                                                        \
  do {                                                                                          \
    if (sparse) reset_sparse_kernel<KIND, CNT_><<<blocks, 256, 0, st>>>(p, mask, e->n_resets);  \
    else reset_kernel<KIND, CNT_><<<blocks, 256, 0, st>>>(p, mask, e->n_resets);                \
  } while (0)
  switch (e->cnt_mode) {
    case CNT_U32: MGYM_RESET(CNT_U32); break;
    case CNT_S16: MGYM_RESET(CNT_S16); break;
    default: MGYM_RESET(CNT_S32); break;  // CNT_S32 and CNT_S32_LAZY share the representation
  }
#undef MGYM_RESET
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

// The step index (Philox counter) and the tile-ticket base are host-side launch parameters that change with
// every call, so a captured launch replayed from a CUDA graph would repeat one step's random draws and find its
// tickets spent.  Refuse capture instead of returning wrong results.
bool is_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &status) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return status != cudaStreamCaptureStatusNone;
}

// `capturable`: the call carries no per-call value when the handle keeps a device clock
int refuse_capture(const mgym_env* e, cudaStream_t st, const char* what, bool capturable) {
  if (!is_capturing(st)) return MGYM_OK;
  if (capturable && e->cfg.device_clock && e->cfg.validate_actions)
    return fail(MGYM_ERR_BAD_ARGUMENT, "%s: validate_actions reads a flag back before every step, which a captured "
                "stream cannot do; create the handle without it", what);
  if (capturable && e->cfg.device_clock) return MGYM_OK;
  if (capturable)
    return fail(MGYM_ERR_BAD_ARGUMENT,
                "%s: the stream is being captured into a CUDA graph; step index and tile tickets are per-call "
                "launch parameters of this handle, a replay would be wrong (create the handle with "
                "device_clock = 1, or use mgym_rollout for fused multi-step launches)",
                what);
  return fail(MGYM_ERR_BAD_ARGUMENT, "%s cannot be captured into a CUDA graph (it synchronises or depends on host state)",
              what);
}

// device clock: enqueue t += dt, ticket base += the tickets this call's TMA launch drew
int advance_clock(mgym_env* e, uint64_t dt, cudaStream_t st, bool fused = false) {
  if (e->cfg.device_clock && !fused) {
    clock_advance_kernel<<<1, 1, 0, st>>>(e->clock, dt, e->call_tickets);
    MGYM_CUDA(cudaGetLastError());
  }
  e->call_tickets = 0;
  e->t += dt;  // host mirror: exact only while no graph replays the call (mgym_step_index reads the device)
  return MGYM_OK;
}

bool is_host_pointer(const void* ptr) {
  cudaPointerAttributes attr{};
  if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return attr.type == cudaMemoryTypeUnregistered || attr.type == cudaMemoryTypeHost;
}

int invalid_action(const mgym_env* e) {
  return fail(MGYM_ERR_INVALID_ACTION,
              "action outside Discrete(%d) (%s): the reference asserts action_space.contains; nothing was stepped",
              kNumActions[e->kind], kNames[e->kind]);
}

// validate_actions (debug mode): the reference asserts BEFORE any mutation (cartpole.rs:252, mountain_car.rs:294),
// so the batch is scanned by a pre-pass and an invalid one returns MGYM_ERR_INVALID_ACTION with the handle
// untouched -- state, counters, statistics and step index are exactly as before the call.  Costs one small
// launch and a stream synchronisation per call.  `count` device actions (Discrete kinds only).
int validate_device_actions(mgym_env* e, const void* actions, uint64_t count, cudaStream_t st) {
  if (!e->cfg.validate_actions || kContinuous[e->kind] || !actions) return MGYM_OK;
  uint64_t blocks = (count + 255) / 256;
  if (blocks > (uint64_t)e->num_sms * 8) blocks = (uint64_t)e->num_sms * 8;
  MGYM_CUDA(cudaMemsetAsync(e->bad_action, 0, sizeof(uint32_t), st));
  validate_actions_kernel<<<(unsigned)blocks, 256, 0, st>>>(static_cast<const uint8_t*>(actions), count,
                                                             (uint32_t)kNumActions[e->kind], e->bad_action);
  MGYM_CUDA(cudaGetLastError());
  uint32_t bad = 0;
  MGYM_CUDA(cudaMemcpyAsync(&bad, e->bad_action, sizeof(bad), cudaMemcpyDeviceToHost, st));
  MGYM_CUDA(cudaStreamSynchronize(st));
  return bad ? invalid_action(e) : MGYM_OK;
}

// Redraw ranges (mgym_set_param_redraw, checkpoints): finite, low <= high, low > 0 for the kind's positive
// parameters.  Names the first offending parameter.
int check_redraw_ranges(int kind, const float* low, const float* high, const char* what) {
  for (int c = 0; c < kNumParams[kind]; ++c) {
    const bool pos = (kParamPositive[kind] >> c) & 1u;
    if (!std::isfinite(low[c]) || !std::isfinite(high[c]) || !(low[c] <= high[c]) || (pos && !(low[c] > 0.0f)))
      return fail(MGYM_ERR_BAD_ARGUMENT, "%s: bad range for %s %s: [%g, %g] (finite, low <= high%s); nothing was changed",
                  what, kNames[kind], kParamNames[kind][c], (double)low[c], (double)high[c], pos ? ", low > 0" : "");
  }
  return MGYM_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// metadata
// ---------------------------------------------------------------------------------------------
extern "C" {

int mgym_abi_version(void) { return MGYM_ABI_VERSION; }
const char* mgym_last_error(void) { return g_last_error.c_str(); }
const char* mgym_kind_name(int kind) { return valid_kind(kind) ? kNames[kind] : "?"; }
int mgym_state_dim(int kind) { return valid_kind(kind) ? kStateDim[kind] : MGYM_ERR_BAD_ARGUMENT; }
int mgym_obs_dim(int kind) { return valid_kind(kind) ? kObsDim[kind] : MGYM_ERR_BAD_ARGUMENT; }
int mgym_action_is_continuous(int kind) { return valid_kind(kind) ? kContinuous[kind] : MGYM_ERR_BAD_ARGUMENT; }
int mgym_num_actions(int kind) { return valid_kind(kind) ? kNumActions[kind] : MGYM_ERR_BAD_ARGUMENT; }

int mgym_space_observation(int kind, float* low, float* high) {
  if (!valid_kind(kind) || !low || !high) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_space_observation: bad argument");
  const float inf = std::numeric_limits<float>::infinity();
  mgym_config cfg{};
  const EnvConsts k = make_consts(kind, cfg);
  switch (kind) {
    case MGYM_CARTPOLE_V1: {  // cartpole.rs:58-64
      volatile float xt = k.x_threshold, tt = k.theta_threshold;
      const float hi[4] = {xt * 2.0f, inf, tt * 2.0f, inf};
      for (int c = 0; c < 4; ++c) high[c] = hi[c], low[c] = -hi[c];
      break;
    }
    case MGYM_MOUNTAIN_CAR_V0:  // mountain_car.rs:42-43
    case MGYM_MOUNTAIN_CAR_CONTINUOUS_V0:
      low[0] = k.min_position, low[1] = -k.max_speed, high[0] = k.max_position, high[1] = k.max_speed;
      break;
    case MGYM_PENDULUM_V1:
      low[0] = low[1] = -1.0f, low[2] = -8.0f, high[0] = high[1] = 1.0f, high[2] = 8.0f;
      break;
    default:
      for (int c = 0; c < 4; ++c) low[c] = -1.0f, high[c] = 1.0f;
      low[4] = -k.max_vel_1, high[4] = k.max_vel_1, low[5] = -k.max_vel_2, high[5] = k.max_vel_2;
  }
  return MGYM_OK;
}

int mgym_space_action(int kind, float* low, float* high) {
  if (!valid_kind(kind) || !low || !high) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_space_action: bad argument");
  if (kind == MGYM_MOUNTAIN_CAR_CONTINUOUS_V0) {
    *low = -1.0f, *high = 1.0f;
  } else if (kind == MGYM_PENDULUM_V1) {
    *low = -2.0f, *high = 2.0f;
  } else {
    *low = 0.0f, *high = (float)(kNumActions[kind] - 1);  // Discrete(n): {0..n-1}
  }
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------------
int mgym_config_default(int kind, mgym_config* cfg) {
  if (!valid_kind(kind) || !cfg) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_config_default: bad argument");
  memset(cfg, 0, sizeof(*cfg));
  cfg->struct_size = sizeof(mgym_config);
  cfg->auto_reset = 1;
  cfg->sutton_barto_reward = 0;  // cartpole.rs:39
  cfg->is_euler = 1;             // cartpole.rs:40
  cfg->goal_velocity = 0.0f;     // mountain_car.rs:33
  cfg->track_stats = 1;
  cfg->validate_actions = 0;
  cfg->env_index_base = 0;
  cfg->device_clock = 0;
  cfg->track_returns = 0;
  switch (kind) {
    case MGYM_MOUNTAIN_CAR_CONTINUOUS_V0: cfg->max_episode_steps = 999; break;
    case MGYM_PENDULUM_V1: cfg->max_episode_steps = 200; break;
    case MGYM_ACROBOT_V1: cfg->max_episode_steps = 500; break;
    default: cfg->max_episode_steps = 0;
  }
  return MGYM_OK;
}

int mgym_destroy(mgym_env* e) {
  if (!e) return MGYM_OK;
  DeviceGuard guard(e->device);
  cudaFree(e->clock);
  cudaFree(e->state);
  cudaFree(e->steps);
  cudaFree(e->sbt);
  cudaFree(e->ep_return);
  cudaFree(e->reset_pool);
  cudaFree(e->stats);
  cudaFree(e->bad_action);
  cudaFree(e->params);
  cudaFree(e->h_actions);
  cudaFree(e->h_obs);
  cudaFree(e->h_reward);
  cudaFree(e->h_flags);
  cudaFree(e->work);
  for (auto& s : e->pipe_stream)
    if (s) cudaStreamDestroy(s);
  for (auto& ev : e->pipe_event)
    if (ev) cudaEventDestroy(ev);
  delete e;
  return MGYM_OK;
}

int mgym_create(int kind, uint64_t num_envs, int device_ordinal, uint64_t seed, const mgym_config* cfg_in,
                mgym_env** out) {
  if (!out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_create: out is NULL");
  *out = nullptr;
  if (!valid_kind(kind)) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_create: unknown kind %d", kind);
  if (num_envs == 0) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_create: num_envs must be > 0");
  mgym_config cfg;
  mgym_config_default(kind, &cfg);
  if (cfg_in) {
    if (cfg_in->struct_size != sizeof(mgym_config))
      return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_create: cfg->struct_size %u != %zu", cfg_in->struct_size,
                  sizeof(mgym_config));
    cfg = *cfg_in;
  }
  if (cfg.max_episode_steps < 0) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_create: max_episode_steps < 0");

  int n_dev = 0;
  cudaError_t ce = cudaGetDeviceCount(&n_dev);
  if (ce != cudaSuccess || n_dev == 0)
    return fail(MGYM_ERR_CUDA, "mgym_create: no CUDA device (%s); there is no CPU fallback",
                ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
  if (device_ordinal < 0 || device_ordinal >= n_dev)
    return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_create: device %d out of range [0,%d)", device_ordinal, n_dev);

  mgym_env* e = new (std::nothrow) mgym_env();
  if (!e) return fail(MGYM_ERR_OUT_OF_MEMORY, "mgym_create: host allocation failed");
  e->kind = kind;
  e->n = num_envs;
  e->device = device_ordinal;
  e->seed = seed;
  e->cfg = cfg;
  e->k = make_consts(kind, cfg);
  e->vec4 = (num_envs % 4 == 0) && (cfg.env_index_base % 4 == 0);

  // counter representation (DESIGN.md section 4, CounterMode in mgym_kernels.cuh)
  if (!cfg.auto_reset) {
    e->cnt_mode = CNT_U32;  // the reference's steps_since_reset (cartpole.rs:24)
  } else if (kind == MGYM_CARTPOLE_V1) {
    e->cnt_mode = CNT_S16;  // <= 500 between resets: a 16-bit start stamp (read-only per step)
  } else if (cfg.max_episode_steps > 0 && cfg.max_episode_steps <= 65535) {
    e->cnt_mode = CNT_S16;
  } else if (cfg.max_episode_steps > 65535) {
    e->cnt_mode = CNT_S32;
  } else {
    // no time limit: only a FINISHED env needs its episode length (it keys the reset stream and feeds the
    // statistics), so the stamp is not touched by a step until then -- MountainCar-v0 moves no counter, like the
    // reference (mountain_car.rs:10-23)
    e->cnt_mode = CNT_S32_LAZY;
  }

  DeviceGuard guard(device_ordinal);
  int rc = [&]() -> int {
    cudaDeviceProp prop;
    MGYM_CUDA(cudaGetDeviceProperties(&prop, device_ordinal));
    e->num_sms = prop.multiProcessorCount;
    const size_t n = (size_t)num_envs;
    MGYM_CUDA(cudaMalloc(&e->state, sizeof(float) * kStateDim[kind] * n));
    MGYM_CUDA(cudaMemset(e->state, 0, sizeof(float) * kStateDim[kind] * n));  // cartpole.rs:85 zero state
    // count 0, or start stamp 0 = the handle's step index right now
    MGYM_CUDA(cudaMalloc(&e->steps, counter_width(e->cnt_mode) * n));
    MGYM_CUDA(cudaMemset(e->steps, 0, counter_width(e->cnt_mode) * n));
    if (!cfg.auto_reset && kind == MGYM_CARTPOLE_V1) {
      MGYM_CUDA(cudaMalloc(&e->sbt, sizeof(uint32_t) * n));
      fill_u32_kernel<<<(unsigned)((n + 255) / 256), 256>>>(e->sbt, 1u, n);  // cartpole.rs:81 Some(0)
      MGYM_CUDA(cudaGetLastError());
    }
    const bool analytic = kind == MGYM_CARTPOLE_V1 || kind == MGYM_MOUNTAIN_CAR_V0 || kind == MGYM_ACROBOT_V1;
    if (cfg.auto_reset && cfg.track_stats && cfg.track_returns && !analytic) {
      MGYM_CUDA(cudaMalloc(&e->ep_return, sizeof(float) * n));
      MGYM_CUDA(cudaMemset(e->ep_return, 0, sizeof(float) * n));
    }
    MGYM_CUDA(cudaMalloc(&e->stats, 5 * sizeof(unsigned long long)));
    MGYM_CUDA(cudaMemset(e->stats, 0, 5 * sizeof(unsigned long long)));
    MGYM_CUDA(cudaMalloc(&e->clock, 3 * sizeof(unsigned long long)));
    MGYM_CUDA(cudaMemset(e->clock, 0, 3 * sizeof(unsigned long long)));
    MGYM_CUDA(cudaMalloc(&e->work, 4 * sizeof(unsigned long long)));
    MGYM_CUDA(cudaMemset(e->work, 0, 4 * sizeof(unsigned long long)));
    MGYM_CUDA(cudaMalloc(&e->bad_action, sizeof(uint32_t)));
    MGYM_CUDA(cudaMemset(e->bad_action, 0, sizeof(uint32_t)));
    MGYM_CUDA(cudaDeviceSynchronize());
    return MGYM_OK;
  }();
  if (rc != MGYM_OK) {
    std::string keep = g_last_error;
    mgym_destroy(e);
    g_last_error = keep;
    return rc;
  }
  *out = e;
  return MGYM_OK;
}

uint64_t mgym_num_envs(const mgym_env* e) { return e ? e->n : 0; }
int mgym_kind_of(const mgym_env* e) { return e ? e->kind : MGYM_ERR_BAD_ARGUMENT; }
// With a device clock the authoritative step index is on the device (graph replays advance it without the
// host's knowledge): this then synchronises the device and refreshes the host mirror.
uint64_t mgym_step_index(const mgym_env* ce) {
  if (!ce) return 0;
  mgym_env* e = const_cast<mgym_env*>(ce);
  if (e->cfg.device_clock) {
    DeviceGuard guard(e->device);
    unsigned long long t = e->t;
    if (cudaDeviceSynchronize() == cudaSuccess &&
        cudaMemcpy(&t, e->clock, sizeof(t), cudaMemcpyDeviceToHost) == cudaSuccess)
      e->t = t;
    else
      cudaGetLastError();
  }
  return e->t;
}
float* mgym_state_ptr(mgym_env* e) { return e ? e->state : nullptr; }

// ---------------------------------------------------------------------------------------------
// reset
// ---------------------------------------------------------------------------------------------
int mgym_reset_masked(mgym_env* e, const uint8_t* mask, float* obs_out, void* stream) {
  if (e) {
    if (int rc = refuse_capture(e, (cudaStream_t)stream, "mgym_reset", false)) return rc;  // reset index is host state
  }
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_reset: env is NULL");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  KernelParams p = base_params(e);
  p.obs_out = obs_out;
  int rc;
  switch (e->kind) {
    case 0: rc = launch_reset_kind<0>(e, p, mask, st); break;
    case 1: rc = launch_reset_kind<1>(e, p, mask, st); break;
    case 2: rc = launch_reset_kind<2>(e, p, mask, st); break;
    case 3: rc = launch_reset_kind<3>(e, p, mask, st); break;
    default: rc = launch_reset_kind<4>(e, p, mask, st); break;
  }
  if (rc == MGYM_OK && e->redraw) {  // the reset envs' parameters, keyed like their reset states
    reset_redraw_params_kernel<<<(unsigned)((e->n + 255) / 256), 256, 0, st>>>(
        e->params, e->n, kNumParams[e->kind], mask, e->seed, e->cfg.env_index_base, e->n_resets, redraw_box(e));
    MGYM_CUDA(cudaGetLastError());
  }
  if (rc == MGYM_OK) e->n_resets += 1;
  return rc;
}

int mgym_reset(mgym_env* e, float* obs_out, void* stream) { return mgym_reset_masked(e, nullptr, obs_out, stream); }

int mgym_set_reset_pool(mgym_env* e, const float* pool, uint64_t pool_len, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_set_reset_pool: env is NULL");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  MGYM_CUDA(cudaStreamSynchronize(st));
  cudaFree(e->reset_pool);
  e->reset_pool = nullptr;
  e->pool_len = 0;
  if (!pool || pool_len == 0) return MGYM_OK;
  const size_t bytes = sizeof(float) * kStateDim[e->kind] * (size_t)pool_len;
  MGYM_CUDA(cudaMalloc(&e->reset_pool, bytes));
  MGYM_CUDA(cudaMemcpyAsync(e->reset_pool, pool, bytes, cudaMemcpyDefault, st));
  MGYM_CUDA(cudaStreamSynchronize(st));
  e->pool_len = pool_len;
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// state injection / checkpoint
// ---------------------------------------------------------------------------------------------
int mgym_set_state(mgym_env* e, const float* state, const uint32_t* steps, const uint32_t* sbt, void* stream) {
  if (!e || !state) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_set_state: NULL argument");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)e->n;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  MGYM_CUDA(cudaMemcpyAsync(e->state, state, sizeof(float) * kStateDim[e->kind] * n, cudaMemcpyDefault, st));
  // the caller's uint32 counts -> this handle's representation (a count, or a start stamp relative to t)
  const uint32_t* src = steps;
  uint32_t* tmp = nullptr;
  if (steps && is_host_pointer(steps)) {  // set_state/get_state also accept host arrays
    MGYM_CUDA(cudaMalloc(&tmp, sizeof(uint32_t) * n));
    MGYM_CUDA(cudaMemcpyAsync(tmp, steps, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, st));
    src = tmp;
  }
  const unsigned long long* td = e->cfg.device_clock ? e->clock : nullptr;
  switch (e->cnt_mode) {
    case CNT_U32: counters_from_steps_kernel<CNT_U32><<<blocks, 256, 0, st>>>(src, (uint32_t*)e->steps, n, e->t, td); break;
    case CNT_S16: counters_from_steps_kernel<CNT_S16><<<blocks, 256, 0, st>>>(src, (uint16_t*)e->steps, n, e->t, td); break;
    default: counters_from_steps_kernel<CNT_S32><<<blocks, 256, 0, st>>>(src, (uint32_t*)e->steps, n, e->t, td); break;
  }
  MGYM_CUDA(cudaGetLastError());
  if (tmp) {
    MGYM_CUDA(cudaStreamSynchronize(st));
    cudaFree(tmp);
  }
  if (e->sbt) {
    if (sbt) MGYM_CUDA(cudaMemcpyAsync(e->sbt, sbt, sizeof(uint32_t) * n, cudaMemcpyDefault, st));
    else MGYM_CUDA(cudaMemsetAsync(e->sbt, 0, sizeof(uint32_t) * n, st));  // None
  }
  if (e->ep_return) MGYM_CUDA(cudaMemsetAsync(e->ep_return, 0, sizeof(float) * n, st));
  return MGYM_OK;
}

int mgym_get_state(mgym_env* e, float* state, uint32_t* steps, uint32_t* sbt, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_get_state: env is NULL");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)e->n;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (state) MGYM_CUDA(cudaMemcpyAsync(state, e->state, sizeof(float) * kStateDim[e->kind] * n, cudaMemcpyDefault, st));
  if (steps) {
    const bool host = is_host_pointer(steps);
    uint32_t* dst = steps;
    uint32_t* tmp = nullptr;
    if (host) {
      MGYM_CUDA(cudaMalloc(&tmp, sizeof(uint32_t) * n));
      dst = tmp;
    }
    const unsigned long long* td = e->cfg.device_clock ? e->clock : nullptr;
    switch (e->cnt_mode) {
      case CNT_U32: steps_from_counters_kernel<CNT_U32><<<blocks, 256, 0, st>>>((const uint32_t*)e->steps, dst, n, e->t, td); break;
      case CNT_S16: steps_from_counters_kernel<CNT_S16><<<blocks, 256, 0, st>>>((const uint16_t*)e->steps, dst, n, e->t, td); break;
      default: steps_from_counters_kernel<CNT_S32><<<blocks, 256, 0, st>>>((const uint32_t*)e->steps, dst, n, e->t, td); break;
    }
    MGYM_CUDA(cudaGetLastError());
    if (host) {
      MGYM_CUDA(cudaMemcpyAsync(steps, tmp, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st));
      MGYM_CUDA(cudaStreamSynchronize(st));
      cudaFree(tmp);
    }
  }
  if (sbt) {
    if (e->sbt) MGYM_CUDA(cudaMemcpyAsync(sbt, e->sbt, sizeof(uint32_t) * n, cudaMemcpyDefault, st));
    else if (is_host_pointer(sbt)) memset(sbt, 0, sizeof(uint32_t) * n);
    else MGYM_CUDA(cudaMemsetAsync(sbt, 0, sizeof(uint32_t) * n, st));
  }
  return MGYM_OK;
}

int mgym_get_obs(mgym_env* e, float* obs_out, void* stream) {
  if (!e || !obs_out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_get_obs: NULL argument");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((e->n + 255) / 256);
  // like the state accessors, this one also takes a HOST array (scalar adapters, tests)
  const bool host = is_host_pointer(obs_out);
  const size_t bytes = sizeof(float) * kObsDim[e->kind] * (size_t)e->n;
  float* dst = obs_out;
  if (host) MGYM_CUDA(cudaMalloc(&dst, bytes));
  switch (e->kind) {
    case 0: obs_kernel<0><<<blocks, 256, 0, st>>>(e->state, dst, e->n); break;
    case 1: obs_kernel<1><<<blocks, 256, 0, st>>>(e->state, dst, e->n); break;
    case 2: obs_kernel<2><<<blocks, 256, 0, st>>>(e->state, dst, e->n); break;
    case 3: obs_kernel<3><<<blocks, 256, 0, st>>>(e->state, dst, e->n); break;
    default: obs_kernel<4><<<blocks, 256, 0, st>>>(e->state, dst, e->n); break;
  }
  cudaError_t err = cudaGetLastError();
  if (host) {
    if (err == cudaSuccess) err = cudaMemcpyAsync(obs_out, dst, bytes, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    cudaFree(dst);
  }
  if (err != cudaSuccess) return fail(MGYM_ERR_CUDA, "mgym_get_obs: %s", cudaGetErrorString(err));
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// checkpoint / resume
// ---------------------------------------------------------------------------------------------
namespace {
// Everything a bit-identical continuation depends on besides the arrays themselves: a blob only loads into a handle
// whose dynamics-relevant configuration matches (the seed, step index and reset index come from the blob).
struct CheckpointHeader {
  uint32_t magic, version;
  int32_t kind, cnt_mode, auto_reset, has_sbt, has_ret;
  int32_t is_euler, sutton_barto, max_episode_steps, track_stats;
  float goal_velocity;
  uint32_t has_params;  // bit 0: the per-env parameter rows follow the statistics; bit 1: the redraw ranges (P low, then
                        // P high values) follow the rows
  uint64_t n, seed, t, n_resets, env_index_base, pool_len;
};
constexpr uint32_t kCkptMagic = 0x4D47594Du;  // "MGYM"
constexpr uint32_t kCkptVersion = 2;

CheckpointHeader checkpoint_header(const mgym_env* e) {
  CheckpointHeader h;
  memset(&h, 0, sizeof(h));  // padding included: blobs are reproducible byte for byte
  h.magic = kCkptMagic, h.version = kCkptVersion;
  h.kind = e->kind, h.cnt_mode = e->cnt_mode, h.auto_reset = e->cfg.auto_reset;
  h.has_sbt = e->sbt ? 1 : 0, h.has_ret = e->ep_return ? 1 : 0;
  h.is_euler = e->cfg.is_euler, h.sutton_barto = e->cfg.sutton_barto_reward;
  h.max_episode_steps = e->cfg.max_episode_steps, h.track_stats = e->cfg.track_stats;
  h.goal_velocity = e->cfg.goal_velocity;
  h.n = e->n, h.seed = e->seed, h.t = e->t, h.n_resets = e->n_resets;
  h.env_index_base = e->cfg.env_index_base, h.pool_len = e->pool_len;
  h.has_params = (e->params ? 1u : 0u) | (e->redraw ? 2u : 0u);
  return h;
}

size_t counter_bytes(const mgym_env* e) { return counter_width(e->cnt_mode) * (size_t)e->n; }
size_t param_bytes(const mgym_env* e) { return sizeof(float) * kNumParams[e->kind] * (size_t)e->n; }
size_t range_bytes(const mgym_env* e) { return 2 * sizeof(float) * kNumParams[e->kind]; }

// size of a blob of this handle that carries parameter rows (and redraw ranges) or not
size_t checkpoint_bytes(const mgym_env* e, bool with_params, bool with_ranges) {
  const size_t n = (size_t)e->n;
  return sizeof(CheckpointHeader) + sizeof(float) * kStateDim[e->kind] * n + counter_bytes(e) +
         (e->sbt ? sizeof(uint32_t) * n : 0) + (e->ep_return ? sizeof(float) * n : 0) + 5 * sizeof(unsigned long long) +
         (with_params ? param_bytes(e) : 0) + (with_ranges ? range_bytes(e) : 0);
}
}  // namespace

size_t mgym_checkpoint_size(const mgym_env* e) {
  return e ? checkpoint_bytes(e, e->params != nullptr, e->redraw) : 0;
}

int mgym_checkpoint_save(mgym_env* e, void* blob, size_t blob_bytes, void* stream) {
  if (!e || !blob) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_save: NULL argument");
  if (blob_bytes < mgym_checkpoint_size(e)) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_save: blob too small");
  (void)mgym_step_index(e);  // device clock: refresh e->t from the device
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)e->n;
  const CheckpointHeader h = checkpoint_header(e);
  uint8_t* out = static_cast<uint8_t*>(blob);
  memcpy(out, &h, sizeof(h));
  out += sizeof(h);
  auto pull = [&](const void* dev, size_t bytes) -> int {
    if (bytes) MGYM_CUDA(cudaMemcpyAsync(out, dev, bytes, cudaMemcpyDeviceToHost, st));
    out += bytes;
    return MGYM_OK;
  };
  int rc;
  if ((rc = pull(e->state, sizeof(float) * kStateDim[e->kind] * n))) return rc;
  if ((rc = pull(e->steps, counter_bytes(e)))) return rc;
  if ((rc = pull(e->sbt, e->sbt ? sizeof(uint32_t) * n : 0))) return rc;
  if ((rc = pull(e->ep_return, e->ep_return ? sizeof(float) * n : 0))) return rc;
  if ((rc = pull(e->stats, 5 * sizeof(unsigned long long)))) return rc;
  if ((rc = pull(e->params, e->params ? param_bytes(e) : 0))) return rc;
  MGYM_CUDA(cudaStreamSynchronize(st));
  if (e->redraw) {
    const size_t np = (size_t)kNumParams[e->kind];
    memcpy(out, e->redraw_lo, sizeof(float) * np);
    memcpy(out + sizeof(float) * np, e->redraw_hi, sizeof(float) * np);
  }
  return MGYM_OK;
}

int mgym_checkpoint_load(mgym_env* e, const void* blob, size_t blob_bytes, void* stream) {
  if (!e || !blob) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_load: NULL argument");
  if (blob_bytes < sizeof(CheckpointHeader)) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_load: truncated blob");
  CheckpointHeader h;
  memcpy(&h, blob, sizeof(h));
  if (h.magic != kCkptMagic || h.version != kCkptVersion)
    return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_load: not a checkpoint of this library version");
  const CheckpointHeader mine = checkpoint_header(e);
  if (h.kind != mine.kind || h.n != mine.n || h.cnt_mode != mine.cnt_mode || h.auto_reset != mine.auto_reset ||
      h.has_sbt != mine.has_sbt || h.has_ret != mine.has_ret)
    return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_load: checkpoint of %s x %llu does not match this handle",
                valid_kind(h.kind) ? kNames[h.kind] : "?", (unsigned long long)h.n);
  if (h.is_euler != mine.is_euler || h.sutton_barto != mine.sutton_barto || h.max_episode_steps != mine.max_episode_steps ||
      h.track_stats != mine.track_stats || memcmp(&h.goal_velocity, &mine.goal_velocity, sizeof(float)) != 0 ||
      h.env_index_base != mine.env_index_base || h.pool_len != mine.pool_len)
    return fail(MGYM_ERR_BAD_ARGUMENT,
                "mgym_checkpoint_load: the checkpoint was taken with a different configuration (is_euler %d/%d, "
                "sutton_barto %d/%d, max_episode_steps %d/%d, track_stats %d/%d, goal_velocity %g/%g, env_index_base "
                "%llu/%llu, reset pool %llu/%llu): the continuation would not be bit-identical",
                h.is_euler, mine.is_euler, h.sutton_barto, mine.sutton_barto, h.max_episode_steps, mine.max_episode_steps,
                h.track_stats, mine.track_stats, (double)h.goal_velocity, (double)mine.goal_velocity,
                (unsigned long long)h.env_index_base, (unsigned long long)mine.env_index_base,
                (unsigned long long)h.pool_len, (unsigned long long)mine.pool_len);
  // a blob restores exactly the parameters it carries; one without parameter rows clears the handle's
  const bool with_params = (h.has_params & 1u) != 0 && kNumParams[e->kind] > 0;
  const bool with_ranges = with_params && (h.has_params & 2u) != 0;
  if (blob_bytes < checkpoint_bytes(e, with_params, with_ranges))
    return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_checkpoint_load: truncated blob");
  float lo[MAX_PARAMS] = {}, hi[MAX_PARAMS] = {};
  if (with_ranges) {  // checked like mgym_set_param_redraw, before anything changes
    const size_t np = (size_t)kNumParams[e->kind];
    const uint8_t* r = static_cast<const uint8_t*>(blob) + checkpoint_bytes(e, true, false);
    memcpy(lo, r, sizeof(float) * np);
    memcpy(hi, r + sizeof(float) * np, sizeof(float) * np);
    if (int rc = check_redraw_ranges(e->kind, lo, hi, "mgym_checkpoint_load")) return rc;
  }
  DeviceGuard guard(e->device);
  if (with_params && !e->params) MGYM_CUDA(cudaMalloc(&e->params, param_bytes(e)));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)e->n;
  const uint8_t* in = static_cast<const uint8_t*>(blob) + sizeof(h);
  auto push = [&](void* dev, size_t bytes) -> int {
    if (bytes) MGYM_CUDA(cudaMemcpyAsync(dev, in, bytes, cudaMemcpyHostToDevice, st));
    in += bytes;
    return MGYM_OK;
  };
  int rc;
  if ((rc = push(e->state, sizeof(float) * kStateDim[e->kind] * n))) return rc;
  if ((rc = push(e->steps, counter_bytes(e)))) return rc;
  if ((rc = push(e->sbt, e->sbt ? sizeof(uint32_t) * n : 0))) return rc;
  if ((rc = push(e->ep_return, e->ep_return ? sizeof(float) * n : 0))) return rc;
  if ((rc = push(e->stats, 5 * sizeof(unsigned long long)))) return rc;
  if ((rc = push(e->params, with_params ? param_bytes(e) : 0))) return rc;
  MGYM_CUDA(cudaStreamSynchronize(st));
  if (!with_params) {
    cudaFree(e->params);
    e->params = nullptr;
  }
  // exactly the ranges the blob carries: a blob without them turns redraw off
  e->redraw = with_ranges;
  memcpy(e->redraw_lo, lo, sizeof(lo));
  memcpy(e->redraw_hi, hi, sizeof(hi));
  e->seed = h.seed;
  e->t = h.t;
  if (e->cfg.device_clock) {
    const unsigned long long t = h.t;
    MGYM_CUDA(cudaMemcpyAsync(e->clock, &t, sizeof(t), cudaMemcpyHostToDevice, st));
    MGYM_CUDA(cudaStreamSynchronize(st));
  }
  e->n_resets = h.n_resets;
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// hot path
// ---------------------------------------------------------------------------------------------
int mgym_step(mgym_env* e, const void* actions, float* obs_out, float* reward_out, uint8_t* flags_out,
              float* final_obs_out, void* stream) {
  if (!e || !actions) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_step: NULL argument");
  e->work_slot = 0;
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = refuse_capture(e, st, "mgym_step", true)) return rc;
  if (int rc = validate_device_actions(e, actions, e->n, st)) return rc;
  e->call_tickets = 0;
  KernelParams p = base_params(e);
  p.actions = actions;
  // zero-copy observation: for kinds whose observation is the state, obs_out == state rows is a no-op
  p.obs_out = (obs_out == e->state) ? nullptr : obs_out;
  p.reward_out = reward_out;
  p.flags_out = flags_out;
  p.final_obs_out = final_obs_out;
  p.adv_clock = e->cfg.device_clock ? e->clock : nullptr;
  p.adv_dt = 1;
  const bool vec4 = e->vec4 && aligned16(actions) && aligned16(obs_out) && aligned16(reward_out) &&
                    aligned16(flags_out) && aligned16(final_obs_out);
  int rc = dispatch<false>(e, p, vec4, st);
  if (rc != MGYM_OK) return rc;
  return advance_clock(e, 1, st, /*fused=*/true);
}

// mgym_rollout and mgym_rollout_final: a non-null final_obs_traj selects the FINAL kernel forms, null launches exactly
// what mgym_rollout launches
static int run_rollout(const char* fn, mgym_env* e, uint32_t K, const void* actions, float* obs_traj, float* reward_traj,
                       uint8_t* flags_traj, float* final_obs_traj, unsigned long long* done_count_out, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "%s: env is NULL", fn);
  if (final_obs_traj) {
    if (!e->cfg.auto_reset)
      return fail(MGYM_ERR_BAD_ARGUMENT, "%s: a manual-mode handle resets nothing inside the rollout; obs_traj "
                  "already holds the final observations", fn);
    if (final_obs_traj == obs_traj)
      return fail(MGYM_ERR_BAD_ARGUMENT, "%s: final_obs_traj must not be obs_traj", fn);
  }
  if (K == 0) return MGYM_OK;
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = refuse_capture(e, st, fn, true)) return rc;
  if (int rc = validate_device_actions(e, actions, (uint64_t)K * e->n, st)) return rc;
  e->call_tickets = 0;
  KernelParams p = base_params(e);
  p.actions = actions;
  p.obs_out = obs_traj;
  p.reward_out = reward_traj;
  p.flags_out = flags_traj;
  p.done_count = done_count_out;
  p.K = K;
  p.adv_clock = e->cfg.device_clock ? e->clock : nullptr;
  p.adv_dt = K;
  if (done_count_out) MGYM_CUDA(cudaMemsetAsync(done_count_out, 0, sizeof(unsigned long long), st));
  const bool vec4 = e->vec4 && aligned16(actions) && aligned16(obs_traj) && aligned16(reward_traj) &&
                    aligned16(flags_traj);
  // warp-tile tickets of this launch start at 0: the rollout has its own counter, cleared in-stream
  p.work_counter = e->work + 3;
  p.work_base = 0;
  MGYM_CUDA(cudaMemsetAsync(e->work + 3, 0, sizeof(unsigned long long), st));
  int rc;
  if (final_obs_traj) {
    p.final_obs_out = final_obs_traj;  // float alignment suffices: stored one scalar at a time
    rc = dispatch<true, true>(e, p, vec4, st);
  } else {
    rc = dispatch<true>(e, p, vec4, st);
  }
  if (rc != MGYM_OK) return rc;
  return advance_clock(e, K, st, /*fused=*/true);
}

int mgym_rollout(mgym_env* e, uint32_t K, const void* actions, float* obs_traj, float* reward_traj,
                 uint8_t* flags_traj, unsigned long long* done_count_out, void* stream) {
  return run_rollout("mgym_rollout", e, K, actions, obs_traj, reward_traj, flags_traj, nullptr, done_count_out, stream);
}

int mgym_rollout_final(mgym_env* e, uint32_t K, const void* actions, float* obs_traj, float* reward_traj,
                       uint8_t* flags_traj, float* final_obs_traj, unsigned long long* done_count_out, void* stream) {
  return run_rollout("mgym_rollout_final", e, K, actions, obs_traj, reward_traj, flags_traj, final_obs_traj,
                 done_count_out, stream);
}

int mgym_sample_actions(mgym_env* e, void* actions_out, void* stream) {
  if (!e || !actions_out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_sample_actions: NULL argument");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = refuse_capture(e, st, "mgym_sample_actions", true)) return rc;
  const unsigned blocks = (unsigned)((e->n + 255) / 256);
  const uint64_t base = e->cfg.env_index_base;
  const unsigned long long* td = e->cfg.device_clock ? e->clock : nullptr;
  switch (e->kind) {
    case 0: sample_actions_kernel<0><<<blocks, 256, 0, st>>>((uint8_t*)actions_out, e->n, e->seed, base, e->t, td); break;
    case 1: sample_actions_kernel<1><<<blocks, 256, 0, st>>>((uint8_t*)actions_out, e->n, e->seed, base, e->t, td); break;
    case 2: sample_actions_kernel<2><<<blocks, 256, 0, st>>>((float*)actions_out, e->n, e->seed, base, e->t, td); break;
    case 3: sample_actions_kernel<3><<<blocks, 256, 0, st>>>((float*)actions_out, e->n, e->seed, base, e->t, td); break;
    default: sample_actions_kernel<4><<<blocks, 256, 0, st>>>((uint8_t*)actions_out, e->n, e->seed, base, e->t, td); break;
  }
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// per-env physics parameters
// ---------------------------------------------------------------------------------------------
int mgym_num_params(int kind) { return valid_kind(kind) ? kNumParams[kind] : MGYM_ERR_BAD_ARGUMENT; }

const char* mgym_param_name(int kind, int i) {
  return (valid_kind(kind) && i >= 0 && i < kNumParams[kind]) ? kParamNames[kind][i] : nullptr;
}

int mgym_param_defaults(int kind, float* out) {
  if (!valid_kind(kind) || !out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_param_defaults: bad argument");
  for (int c = 0; c < kNumParams[kind]; ++c) out[c] = kParamDefaults[kind][c];
  return MGYM_OK;
}

namespace {
int no_params(const mgym_env* e, const char* what) {
  return fail(MGYM_ERR_BAD_ARGUMENT,
              "%s: %s has no per-env parameters (its RK4 runs on constants folded on the host; see DESIGN.md)", what,
              kNames[e->kind]);
}
ParamVec param_defaults(int kind) {
  ParamVec d{};
  for (int c = 0; c < kNumParams[kind]; ++c) d.v[c] = kParamDefaults[kind][c];
  return d;
}
// the handle's parameter rows, allocated and filled with the defaults on first use
int ensure_params(mgym_env* e, cudaStream_t st) {
  if (e->params) return MGYM_OK;
  float* rows = nullptr;
  MGYM_CUDA(cudaMalloc(&rows, param_bytes(e)));
  fill_params_kernel<<<(unsigned)((e->n + 255) / 256), 256, 0, st>>>(rows, e->n, kNumParams[e->kind],
                                                                     param_defaults(e->kind));
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    cudaFree(rows);
    return fail(MGYM_ERR_CUDA, "ensure_params: %s", cudaGetErrorString(err));
  }
  e->params = rows;
  return MGYM_OK;
}
}  // namespace

int mgym_set_params(mgym_env* e, const float* params, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_set_params: env is NULL");
  if (kNumParams[e->kind] == 0) return no_params(e, "mgym_set_params");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = refuse_capture(e, st, "mgym_set_params", false)) return rc;
  MGYM_CUDA(cudaStreamSynchronize(st));  // in-flight launches may still read the rows
  if (!params) {  // back to the constants: the redraw ranges go with the rows
    cudaFree(e->params);
    e->params = nullptr;
    e->redraw = false;
    return MGYM_OK;
  }
  const int np = kNumParams[e->kind];
  const uint64_t n = e->n;
  // the "must hold" conditions, checked before anything is copied: a rejected set leaves the handle untouched
  bool bad = false;
  if (is_host_pointer(params)) {  // host rows are scanned on the host, as mgym_step_host scans host actions
    for (uint64_t i = 0; i < (uint64_t)np * n && !bad; ++i) {
      const float x = params[i];
      bad = !std::isfinite(x) || (((kParamPositive[e->kind] >> (i / n)) & 1u) && !(x > 0.0f));
    }
  } else {
    uint64_t blocks = ((uint64_t)np * n + 255) / 256;
    if (blocks > (uint64_t)e->num_sms * 8) blocks = (uint64_t)e->num_sms * 8;
    MGYM_CUDA(cudaMemsetAsync(e->bad_action, 0, sizeof(uint32_t), st));
    validate_params_kernel<<<(unsigned)blocks, 256, 0, st>>>(params, n, np, kParamPositive[e->kind], e->bad_action);
    MGYM_CUDA(cudaGetLastError());
    uint32_t flag = 0;
    MGYM_CUDA(cudaMemcpyAsync(&flag, e->bad_action, sizeof(flag), cudaMemcpyDeviceToHost, st));
    MGYM_CUDA(cudaStreamSynchronize(st));
    bad = flag != 0;
  }
  if (bad)
    return fail(MGYM_ERR_BAD_ARGUMENT,
                "mgym_set_params: a %s parameter is not finite, or a mass, length or time step is not > 0; nothing "
                "was changed", kNames[e->kind]);
  if (!e->params) MGYM_CUDA(cudaMalloc(&e->params, param_bytes(e)));
  MGYM_CUDA(cudaMemcpyAsync(e->params, params, param_bytes(e), cudaMemcpyDefault, st));
  MGYM_CUDA(cudaStreamSynchronize(st));
  return MGYM_OK;
}

int mgym_get_params(mgym_env* e, float* out, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_get_params: env is NULL");
  if (kNumParams[e->kind] == 0) return MGYM_OK;  // nothing to write
  if (!out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_get_params: out is NULL");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int np = kNumParams[e->kind];
  const bool host = is_host_pointer(out);
  if (e->params) {
    MGYM_CUDA(cudaMemcpyAsync(out, e->params, param_bytes(e), cudaMemcpyDefault, st));
    if (host) MGYM_CUDA(cudaStreamSynchronize(st));
  } else if (host) {
    for (int c = 0; c < np; ++c)
      for (uint64_t i = 0; i < e->n; ++i) out[(uint64_t)c * e->n + i] = kParamDefaults[e->kind][c];
  } else {
    fill_params_kernel<<<(unsigned)((e->n + 255) / 256), 256, 0, st>>>(out, e->n, np, param_defaults(e->kind));
    MGYM_CUDA(cudaGetLastError());
  }
  return MGYM_OK;
}

int mgym_sample_params(mgym_env* e, const float* low, const float* high, const uint8_t* mask, uint64_t key,
                       void* stream) {
  if (!e || !low || !high) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_sample_params: NULL argument");
  if (kNumParams[e->kind] == 0) return no_params(e, "mgym_sample_params");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int np = kNumParams[e->kind];
  ParamBox box{};
  for (int c = 0; c < np; ++c) {
    const bool pos = (kParamPositive[e->kind] >> c) & 1u;
    if (!std::isfinite(low[c]) || !std::isfinite(high[c]) || !(low[c] <= high[c]) || (pos && !(low[c] > 0.0f)))
      return fail(MGYM_ERR_BAD_ARGUMENT,
                  "mgym_sample_params: bad range for %s %s: [%g, %g] (finite, low <= high%s)", kNames[e->kind],
                  kParamNames[e->kind][c], (double)low[c], (double)high[c], pos ? ", low > 0" : "");
    box.lo[c] = (double)low[c];
    box.range[c] = (double)high[c] - (double)low[c];
  }
  // capturable: the key is the caller's launch argument, nothing depends on host state once the rows exist
  if (!e->params && is_capturing(st))
    return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_sample_params: set or sample the parameters once before capturing "
                "(the rows are allocated on first use)");
  if (int rc = ensure_params(e, st)) return rc;
  sample_params_kernel<<<(unsigned)((e->n + 255) / 256), 256, 0, st>>>(e->params, e->n, np, mask, e->seed,
                                                                       e->cfg.env_index_base, key, box);
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

int mgym_set_param_redraw(mgym_env* e, const float* low, const float* high, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_set_param_redraw: env is NULL");
  if (kNumParams[e->kind] == 0) return no_params(e, "mgym_set_param_redraw");
  if (!low != !high)
    return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_set_param_redraw: low and high must both be given, or both be NULL");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = refuse_capture(e, st, "mgym_set_param_redraw", false)) return rc;
  if (!low) {
    e->redraw = false;
    return MGYM_OK;
  }
  if (int rc = check_redraw_ranges(e->kind, low, high, "mgym_set_param_redraw")) return rc;
  if (int rc = ensure_params(e, st)) return rc;  // rows with the defaults: the current episodes keep their constants
  for (int c = 0; c < MAX_PARAMS; ++c) {
    e->redraw_lo[c] = c < kNumParams[e->kind] ? low[c] : 0.0f;
    e->redraw_hi[c] = c < kNumParams[e->kind] ? high[c] : 0.0f;
  }
  e->redraw = true;
  return MGYM_OK;
}

int mgym_get_param_redraw(const mgym_env* e, int* enabled, float* low, float* high) {
  if (!e || !enabled) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_get_param_redraw: NULL argument");
  *enabled = e->redraw ? 1 : 0;
  for (int c = 0; e->redraw && c < kNumParams[e->kind]; ++c) {
    if (low) low[c] = e->redraw_lo[c];
    if (high) high[c] = e->redraw_hi[c];
  }
  return MGYM_OK;
}

// Host-buffer step.  Large batches are cut into chunks of whole 1024-env tiles that alternate between two
// internal streams, so the D2H of chunk c overlaps the H2D and the kernel of chunk c+1 (PCIe is full duplex):
// the call then costs about the D2H time alone.  Every chunk is one sub-range launch of the ordinary step.
int mgym_step_host(mgym_env* e, const void* actions_host, float* obs_host, float* reward_host, uint8_t* flags_host,
                   void* stream) {
  if (!e || !actions_host) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_step_host: NULL argument");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = refuse_capture(e, st, "mgym_step_host", false)) return rc;
  e->call_tickets = 0;
  const size_t n = (size_t)e->n;
  if (e->cfg.validate_actions && !kContinuous[e->kind]) {  // host actions: scanned on the host, before anything moves
    const uint8_t* a = static_cast<const uint8_t*>(actions_host);
    const uint8_t lim = (uint8_t)kNumActions[e->kind];
    for (size_t i = 0; i < n; ++i)
      if (a[i] >= lim) return invalid_action(e);
  }
  const int od = kObsDim[e->kind];
  const size_t act = action_size(e->kind), asz = act * n, osz = sizeof(float) * od * n;
  const bool obs_is_state = kObsDim[e->kind] == kStateDim[e->kind];
  if (!e->h_actions) MGYM_CUDA(cudaMalloc(&e->h_actions, asz));
  if (obs_host && !obs_is_state && !e->h_obs) MGYM_CUDA(cudaMalloc(&e->h_obs, osz));
  if (reward_host && !e->h_reward) MGYM_CUDA(cudaMalloc(&e->h_reward, sizeof(float) * n));
  if (flags_host && !e->h_flags) MGYM_CUDA(cudaMalloc(&e->h_flags, n));
  // observations of obs-is-state kinds are read straight out of the resident state rows
  float* dev_obs = obs_host ? (obs_is_state ? e->state : e->h_obs) : nullptr;

  constexpr size_t kMinChunk = 1u << 18;  // envs; below 2 chunks the plain path is used
  const size_t chunks = (n >= 2 * kMinChunk && e->vec4) ? (n / kMinChunk > 8 ? 8 : n / kMinChunk) : 1;
  if (chunks > 1 && !e->pipe_stream[0]) {
    for (auto& s : e->pipe_stream) MGYM_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto& ev : e->pipe_event) MGYM_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
  if (chunks > 1) {
    MGYM_CUDA(cudaEventRecord(e->pipe_event[2], st));
    for (auto& s : e->pipe_stream) MGYM_CUDA(cudaStreamWaitEvent(s, e->pipe_event[2], 0));
  }
  const size_t per = ((n / chunks) / TMA_TILE) * TMA_TILE;
  for (size_t c = 0; c < chunks; ++c) {
    cudaStream_t cs = chunks > 1 ? e->pipe_stream[c & 1] : st;
    e->work_slot = chunks > 1 ? 1 + (int)(c & 1) : 0;
    const size_t b = c * per, cnt = (c + 1 == chunks) ? n - b : per;
    MGYM_CUDA(cudaMemcpyAsync((uint8_t*)e->h_actions + act * b, (const uint8_t*)actions_host + act * b, act * cnt,
                              cudaMemcpyHostToDevice, cs));
    KernelParams p = base_params(e);
    p.first = b;
    p.n = cnt;
    p.actions = e->h_actions;
    p.obs_out = (obs_host && !obs_is_state) ? e->h_obs : nullptr;
    p.reward_out = reward_host ? e->h_reward : nullptr;
    p.flags_out = flags_host ? e->h_flags : nullptr;
    int rc = dispatch<false>(e, p, e->vec4, cs);
    if (rc != MGYM_OK) return rc;
    if (obs_host)  // all od rows of this chunk as ONE strided copy (fewer copy-engine round trips than od copies)
      MGYM_CUDA(cudaMemcpy2DAsync(obs_host + b, sizeof(float) * n, dev_obs + b, sizeof(float) * n, sizeof(float) * cnt,
                                  (size_t)od, cudaMemcpyDeviceToHost, cs));
    if (reward_host)
      MGYM_CUDA(cudaMemcpyAsync(reward_host + b, e->h_reward + b, sizeof(float) * cnt, cudaMemcpyDeviceToHost, cs));
    if (flags_host) MGYM_CUDA(cudaMemcpyAsync(flags_host + b, e->h_flags + b, cnt, cudaMemcpyDeviceToHost, cs));
  }
  if (chunks > 1) {
    for (int i = 0; i < 2; ++i) {
      MGYM_CUDA(cudaEventRecord(e->pipe_event[i], e->pipe_stream[i]));
      MGYM_CUDA(cudaStreamWaitEvent(st, e->pipe_event[i], 0));
    }
  }
  e->work_slot = 0;
  if (int rc = advance_clock(e, 1, st)) return rc;
  MGYM_CUDA(cudaStreamSynchronize(st));
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// statistics
// ---------------------------------------------------------------------------------------------
int mgym_stats_get(mgym_env* e, mgym_stats_t* out, void* stream) {
  if (!e || !out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_stats_get: NULL argument");
  DeviceGuard guard(e->device);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long raw[5];
  MGYM_CUDA(cudaMemcpyAsync(raw, e->stats, sizeof(raw), cudaMemcpyDeviceToHost, st));
  MGYM_CUDA(cudaStreamSynchronize(st));
  out->episodes = raw[0];
  out->terminated = raw[1];
  out->truncated = raw[2];
  out->length_sum = raw[3];
  memcpy(&out->return_sum, &raw[4], sizeof(double));
  return MGYM_OK;
}

int mgym_stats_reset(mgym_env* e, void* stream) {
  if (!e) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_stats_reset: env is NULL");
  DeviceGuard guard(e->device);
  MGYM_CUDA(cudaMemsetAsync(e->stats, 0, 5 * sizeof(unsigned long long), (cudaStream_t)stream));
  return MGYM_OK;
}

int mgym_stats_export(mgym_env* e, double* device_vec5_out, void* stream) {
  if (!e || !device_vec5_out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_stats_export: NULL argument");
  DeviceGuard guard(e->device);
  stats_export_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(e->stats, device_vec5_out);
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

int mgym_stats_allreduce(mgym_env* e, void* nccl_comm, double* device_vec5_out, void* stream) {
  if (!e || !nccl_comm || !device_vec5_out) return fail(MGYM_ERR_BAD_ARGUMENT, "mgym_stats_allreduce: NULL argument");
  // ncclResult_t ncclAllReduce(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t)
  using allreduce_fn = int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t);
  static allreduce_fn fn = [] {
    void* sym = dlsym(RTLD_DEFAULT, "ncclAllReduce");
    if (!sym) {
      void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (h) sym = dlsym(h, "ncclAllReduce");
    }
    return reinterpret_cast<allreduce_fn>(sym);
  }();
  if (!fn) return fail(MGYM_ERR_NCCL, "mgym_stats_allreduce: ncclAllReduce not found in this process or libnccl.so.2");
  int rc = mgym_stats_export(e, device_vec5_out, stream);
  if (rc != MGYM_OK) return rc;
  DeviceGuard guard(e->device);
  const int nrc = fn(device_vec5_out, device_vec5_out, 5, kNcclFloat64, kNcclSum, nccl_comm, (cudaStream_t)stream);
  if (nrc != 0) return fail(MGYM_ERR_NCCL, "ncclAllReduce returned %d", nrc);
  return MGYM_OK;
}

// ---------------------------------------------------------------------------------------------
// test probes (not part of include/mgym.h): device sin/cos and Philox for the parity tests
// ---------------------------------------------------------------------------------------------
int mgym_probe_trig(const float* x, float* s, float* c, float* s_only, float* c_only, uint64_t n, void* stream) {
  trig_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, s, c, s_only, c_only, n);
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

// mode 0/1/2 of fast_exhaustive_kernel over bit patterns [first, first+n); out = {checked, bad, first_bad}
int mgym_probe_fast_exhaustive(int mode, uint64_t first, uint64_t n, uint64_t* out3) {
  unsigned long long* d = nullptr;
  MGYM_CUDA(cudaMalloc(&d, 3 * sizeof(unsigned long long)));
  MGYM_CUDA(cudaMemset(d, 0, 2 * sizeof(unsigned long long)));
  MGYM_CUDA(cudaMemset(d + 2, 0xff, sizeof(unsigned long long)));
  mgym_config cfg{};
  const EnvConsts k = make_consts(0, cfg);
  fast_exhaustive_kernel<<<148 * 8, 256>>>(mode, first, n, k.total_mass, k.rcp_total_mass, d, d + 1,
                                           reinterpret_cast<uint32_t*>(d + 2));
  MGYM_CUDA(cudaGetLastError());
  unsigned long long h[3];
  MGYM_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(d);
  out3[0] = h[0], out3[1] = h[1], out3[2] = (uint32_t)h[2];
  return MGYM_OK;
}

int mgym_probe_fast_div_random(uint64_t seed, uint64_t n, uint64_t* out2) {
  unsigned long long* d = nullptr;
  MGYM_CUDA(cudaMalloc(&d, 2 * sizeof(unsigned long long)));
  MGYM_CUDA(cudaMemset(d, 0, 2 * sizeof(unsigned long long)));
  fast_div_random_kernel<<<148 * 8, 256>>>(seed, n, d, d + 1);
  MGYM_CUDA(cudaGetLastError());
  unsigned long long h[2];
  MGYM_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(d);
  out2[0] = h[0], out2[1] = h[1];
  return MGYM_OK;
}

int mgym_probe_cartpole_fast(uint64_t seed, uint64_t n, uint64_t* out3) {
  unsigned long long* d = nullptr;
  MGYM_CUDA(cudaMalloc(&d, 3 * sizeof(unsigned long long)));
  MGYM_CUDA(cudaMemset(d, 0, 3 * sizeof(unsigned long long)));
  mgym_config cfg;
  mgym_config_default(MGYM_CARTPOLE_V1, &cfg);
  cartpole_fast_random_kernel<<<148 * 8, 256>>>(seed, n, make_consts(MGYM_CARTPOLE_V1, cfg), d);
  MGYM_CUDA(cudaGetLastError());
  unsigned long long h[3];
  MGYM_CUDA(cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(d);
  out3[0] = h[0], out3[1] = h[1], out3[2] = h[2];
  return MGYM_OK;
}

int mgym_probe_trig_checksum(uint32_t first, uint64_t count, uint32_t stride, uint64_t* out) {
  unsigned long long* d = nullptr;
  MGYM_CUDA(cudaMalloc(&d, sizeof(unsigned long long)));
  MGYM_CUDA(cudaMemset(d, 0, sizeof(unsigned long long)));
  trig_checksum_kernel<<<148 * 8, 256>>>(first, count, stride, d);
  MGYM_CUDA(cudaGetLastError());
  unsigned long long h = 0;
  MGYM_CUDA(cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(d);
  *out = h;
  return MGYM_OK;
}

int mgym_probe_philox(const uint32_t* ctr_key, uint32_t* out, uint64_t n, void* stream) {
  philox_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ctr_key, out, n);
  MGYM_CUDA(cudaGetLastError());
  return MGYM_OK;
}

}  // extern "C"
