// mgym_kernels.cuh -- the two kernel modes of the hot path.
//
//   step_kernel_tma one Gym::step per env per launch, the headline form: a producer warp stages 1024-env
//                   tiles (state rows, actions, counters) into a shared-memory ring with cp.async.bulk,
//                   eight consumer warps step 4 consecutive envs per thread and store with 128-bit
//                   stores, a reset warp draws the reset states of the envs that finished.  HBM-bound
//                   (profiles/README.md).  Auto-reset and manual (the reference's protocol) forms.
//   step_kernel     the same step with plain vector loads: ragged N (scalar lanes, sub-tile tails),
//                   unaligned buffers.
//   rollout_kernel  K fused steps: state and counters stay in registers, only the trajectory
//                   (obs / reward / flags) is written, actions are read or drawn from Philox.
//
// All are persistent kernels (grid sized from the SM count) so the episode statistics reduce to one
// set of atomics per CTA.  The per-env work is shared: step_group().
#pragma once

#include <type_traits>

#include "mgym_device.cuh"

namespace mgym {

// cp.async (LDGSTS): global -> shared without passing through registers; completion is tracked per thread in
// commit groups.  BYTES = 4 (uint8 x 4 actions) or 16 (float x 4).
template <int BYTES>
__device__ __forceinline__ void cp_async(uint32_t smem_dst, const void* gsrc) {
  static_assert(BYTES == 4 || BYTES == 16, "one lane's four actions");
  if constexpr (BYTES == 16) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
  } else {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(gsrc) : "memory");
  }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory");
}

// Per-env episode step count, as the handle keeps it between launches.  Every handle keeps one: an auto-reset
// handle needs the length of a finished episode (it keys the reset stream, see reset_pending), a manual one keeps the
// reference's counters.
//   CNT_U32       the count itself, read AND written by every step (manual mode = the reference's steps_since_reset,
//                 cartpole.rs:24)
//   CNT_S16/S32   a START STAMP: the handle's step index t at which the episode began (mod 2^16 / 2^32).  The count is
//                 (t - stamp), so a step only READS the stamp; it is written when an episode ends (by the lane that
//                 owns the finished env) -- 2 or 4 bytes read per env-step instead of a read and a write.
//   CNT_S32_LAZY  the same stamp for kinds without a time limit, where only a FINISHED env needs its episode length
//                 (statistics, reset stream): not even read by a step unless the env finished (MountainCar-v0: 22 B per env-step,
//                 the SURVEY 8(d) contract figure, instead of 30).  Kernels that keep the count in registers anyway
//                 (rollout, the LDG step form) treat it as CNT_S32.
// The values are stored in checkpoints (the header's cnt_mode): never renumber them.
enum CounterMode : int { CNT_U32 = 2, CNT_S16 = 3, CNT_S32 = 4, CNT_S32_LAZY = 5 };
__host__ __device__ constexpr bool cnt_is_stamp(int c) { return c >= CNT_S16; }
__host__ __device__ constexpr bool cnt_is_lazy(int c) { return c == CNT_S32_LAZY; }
__host__ __device__ constexpr bool cnt_staged(int c) { return c != CNT_S32_LAZY; }  // read by every step

struct KernelParams {
  // resident env state (owned by the handle)
  float* state;        // [SD][n]
  void* steps;         // uint16_t[n] or uint32_t[n], see CounterMode
  uint32_t* sbt;       // manual CartPole only: steps_beyond_terminated (0 = None, k+1 = Some(k))
  float* ep_return;    // per-env running return (kinds without an analytic return), or null
  // caller buffers
  const void* actions;  // step: [n]; rollout: [K][n] or null (device policy)
  float* obs_out;       // step: [OD][n]; rollout: [K][OD][n]
  float* reward_out;    // step: [n];     rollout: [K][n]
  uint8_t* flags_out;   // step: [n];     rollout: [K][n]
  float* final_obs_out; // step: pre-reset observation [OD][n]; rollout (FINAL forms): [K][OD][n], finished envs only
  // reset source
  const float* reset_pool;  // [SD][pool_len] or null
  uint64_t pool_len;
  // statistics: u64 {episodes, terminated, truncated, length_sum}, then double return_sum
  unsigned long long* stats;
  unsigned long long* done_count;  // rollout: finished env-steps
  unsigned long long* work_counter;  // TMA step kernel: tile tickets (monotonic across launches)
  uint64_t work_base;                // first ticket of this launch
  // Device clock (handles created with device_clock = 1, the CUDA-graph-capturable mode): the step index and
  // the first ticket live in device memory and are advanced by clock_advance_kernel after every call, so a
  // captured launch carries no per-call value.  Null = use `t` / `work_base` above.
  const unsigned long long* t_dev;
  const unsigned long long* base_dev;
  // Fused advance of that clock: the last CTA of the launch to finish adds adv_dt / adv_tickets (every CTA
  // has read the clock by then; the next launch reads it only after this grid has completed).  clock[2] counts
  // finished CTAs.  Null = the host enqueues clock_advance_kernel instead (mgym_step_host's chunked launches).
  unsigned long long* adv_clock;
  uint64_t adv_dt, adv_tickets;
  uint64_t n;      // envs covered by this launch
  uint64_t first;  // index (within the handle) of the first of them
  uint64_t ld;     // row stride of every SoA buffer = envs in the handle
  uint64_t seed, env_base, t;
  uint32_t K;
  PhiloxKeys keys;  // round keys of `seed`
  EnvConsts k;
};
// The launch parameters of the kernels instantiated with PARAMS: the handle's per-env physics parameters [NP][ld]
// (mgym_set_params) on top.  A separate type, so that KernelParams -- and every kernel that takes it by value,
// with the arguments after it -- stays exactly as it is.
struct KernelParamsP : KernelParams {
  const float* params;
};
constexpr int MAX_PARAMS = 8;
struct ParamBox {  // U[lo, lo + range) per parameter, in f64 like the reset draws
  double lo[MAX_PARAMS], range[MAX_PARAMS];
};
// The launch parameters of the kernels instantiated with REDRAW (auto-reset forms only): the handle's redraw ranges
// (mgym_set_param_redraw), by value, on top of the rows -- every auto-reset then writes the new episode's parameters
// into the rows.  A captured launch replays the ranges it was captured with.
struct KernelParamsR : KernelParamsP {
  ParamBox redraw;
};
template <bool PARAMS, bool REDRAW = false>
using KParams = std::conditional_t<REDRAW, KernelParamsR, std::conditional_t<PARAMS, KernelParamsP, KernelParams>>;

// The parameters of global env g for the episode whose reset state has counter (g, t): word c % 4 of the Philox
// block (g, t) with tag tag0 + c / 4, mapped to U[lo, lo + range) as mgym_sample_params maps them.  Parameter c is
// stored to dst[c * stride].
template <int NP>
__device__ __forceinline__ void redraw_params(const PhiloxKeys& ks, const ParamBox& box, uint64_t g, uint64_t t,
                                              uint32_t tag0, float* dst, uint64_t stride) {
#pragma unroll
  for (int b = 0; b * 4 < NP; ++b) {
    const uint4 w = philox_env(ks, g, t, tag0 + (uint32_t)b);
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int j = 0; j < 4 && 4 * b + j < NP; ++j)
      dst[(uint64_t)(4 * b + j) * stride] = uniform_f64_to_f32(ws[j], box.lo[4 * b + j], box.range[4 * b + j]);
  }
}
// Where redraw_pending puts the redrawn parameters: parameter c of slot v at base[c * cstride + v * vstride]
// (the parameter rows in global memory for the per-call step, the per-thread shared-memory slots in the rollout).
struct RedrawDst {
  float* base;
  uint64_t cstride, vstride;
};

// The per-env parameters of a lane's V envs, [NP][V] (r[c][v] = parameter c of slot v).  NP = 0: none.
template <int NP_, int V>
struct ParamRows {
  static constexpr int NP = NP_;
  float r[NP_ > 0 ? NP_ : 1][V];
};
using NoParams = ParamRows<0, 1>;

__device__ __forceinline__ uint64_t launch_t(const KernelParams& p) { return p.t_dev ? *p.t_dev : p.t; }
__device__ __forceinline__ uint64_t launch_work_base(const KernelParams& p) {
  return p.base_dev ? *p.base_dev : p.work_base;
}

// call after the CTA's last use of the clock (all threads may call; thread 0 acts)
__device__ __forceinline__ void fused_clock_advance(const KernelParams& p) {
  if (p.adv_clock && threadIdx.x == 0) {
    const unsigned long long done = atomicAdd(p.adv_clock + 2, 1ull) + 1ull;
    if (done == gridDim.x) {
      p.adv_clock[2] = 0ull;
      p.adv_clock[0] += p.adv_dt;
      p.adv_clock[1] += p.adv_tickets;
    }
  }
}

// ---- vector load/store of V consecutive elements --------------------------------------
template <typename T, int V>
struct Vec {
  T v[V];
};

template <typename T, int V>
__device__ __forceinline__ Vec<T, V> ldv(const T* p) {
  Vec<T, V> r;
  if constexpr (V == 1) {
    r.v[0] = *p;
  } else if constexpr (sizeof(T) * V == 16) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    *reinterpret_cast<uint4*>(&r) = u;
  } else if constexpr (sizeof(T) * V == 8) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    *reinterpret_cast<uint2*>(&r) = u;
  } else {
    static_assert(sizeof(T) * V == 4, "unsupported vector width");
    const uint32_t u = *reinterpret_cast<const uint32_t*>(p);
    *reinterpret_cast<uint32_t*>(&r) = u;
  }
  return r;
}

template <typename T, int V>
__device__ __forceinline__ void stv(T* p, const Vec<T, V>& r) {
  if constexpr (V == 1) {
    *p = r.v[0];
  } else if constexpr (sizeof(T) * V == 16) {
    *reinterpret_cast<uint4*>(p) = *reinterpret_cast<const uint4*>(&r);
  } else if constexpr (sizeof(T) * V == 8) {
    *reinterpret_cast<uint2*>(p) = *reinterpret_cast<const uint2*>(&r);
  } else {
    static_assert(sizeof(T) * V == 4, "unsupported vector width");
    *reinterpret_cast<uint32_t*>(p) = *reinterpret_cast<const uint32_t*>(&r);
  }
}

// ---- actions of V envs kept as the raw loaded word(s), unpacked only where they are used, so a
// prefetched load can stay in flight across a whole rollout step -----------------------------------
template <typename T, int V>
struct RawActions {
  Vec<T, V> v;
  __device__ __forceinline__ void load(const T* p) { v = ldv<T, V>(p); }
  __device__ __forceinline__ void load_shared(uint32_t addr) {
    static_assert(sizeof(T) * V == 16 || V == 1, "one 128-bit shared load");
    if constexpr (V == 1) {
      asm volatile("ld.shared.b32 %0, [%1];" : "=r"(*reinterpret_cast<uint32_t*>(&v.v[0])) : "r"(addr));
    } else {
      uint4 u;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr));
      *reinterpret_cast<uint4*>(&v) = u;
    }
  }
  __device__ __forceinline__ void zero() {
#pragma unroll
    for (int i = 0; i < V; ++i) v.v[i] = T(0);
  }
  __device__ __forceinline__ T get(int i) const { return v.v[i]; }
};
template <>
struct RawActions<uint8_t, 4> {
  uint32_t w;
  __device__ __forceinline__ void load(const uint8_t* p) { w = *reinterpret_cast<const uint32_t*>(p); }
  __device__ __forceinline__ void load_shared(uint32_t addr) { asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(addr)); }
  __device__ __forceinline__ void zero() { w = 0; }
  __device__ __forceinline__ uint8_t get(int i) const { return (uint8_t)(w >> (8 * i)); }
};

// ---- per-thread episode statistics, reduced once per CTA ---------------------------------
struct StatAcc {
  uint32_t episodes = 0, terminated = 0, truncated = 0;
  unsigned long long length_sum = 0;
  double return_sum = 0.0;  // only kinds without an analytic return accumulate here
  unsigned long long done_steps = 0;
};

// Sum of episode returns from the integer sums, for kinds whose rewards are constants.
template <int KIND>
__device__ __forceinline__ double analytic_return_sum(const EnvConsts& k, double episodes, double terminated,
                                                      double truncated, double length_sum) {
  if constexpr (KIND == 0) {  // cartpole.rs:310-347: +1 per step; sutton_barto: -1 on the fall, +1 on truncation
    return k.sutton_barto ? (truncated - terminated) : length_sum;
  } else if constexpr (KIND == 1) {  // mountain_car.rs:319: -1 per step
    return -length_sum;
  } else if constexpr (KIND == 4) {  // Acrobot: -1 per step, 0 on the terminating step
    return terminated - length_sum;
  } else {
    return 0.0 * episodes;
  }
}

template <int KIND>
__device__ __forceinline__ void stats_flush(const StatAcc& a, const KernelParams& p) {
  __shared__ unsigned long long sh_u[5];
  __shared__ double sh_d;
  if (threadIdx.x == 0) {
    sh_u[0] = sh_u[1] = sh_u[2] = sh_u[3] = sh_u[4] = 0ull;
    sh_d = 0.0;
  }
  __syncthreads();
  unsigned long long u0 = a.episodes, u1 = a.terminated, u2 = a.truncated, u3 = a.length_sum, u4 = a.done_steps;
  double d = a.return_sum;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    u0 += __shfl_xor_sync(0xffffffffu, u0, o);
    u1 += __shfl_xor_sync(0xffffffffu, u1, o);
    u2 += __shfl_xor_sync(0xffffffffu, u2, o);
    u3 += __shfl_xor_sync(0xffffffffu, u3, o);
    u4 += __shfl_xor_sync(0xffffffffu, u4, o);
    d += __shfl_xor_sync(0xffffffffu, d, o);
  }
  if ((threadIdx.x & 31) == 0 && (u0 | u4)) {
    atomicAdd(&sh_u[0], u0);
    atomicAdd(&sh_u[1], u1);
    atomicAdd(&sh_u[2], u2);
    atomicAdd(&sh_u[3], u3);
    atomicAdd(&sh_u[4], u4);
    atomicAdd(&sh_d, d);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (p.stats && sh_u[0]) {
      atomicAdd(&p.stats[0], sh_u[0]);
      atomicAdd(&p.stats[1], sh_u[1]);
      atomicAdd(&p.stats[2], sh_u[2]);
      atomicAdd(&p.stats[3], sh_u[3]);
      const double ret = Env<KIND>::ANALYTIC_RETURN
                             ? analytic_return_sum<KIND>(p.k, (double)sh_u[0], (double)sh_u[1], (double)sh_u[2],
                                                         (double)sh_u[3])
                             : sh_d;
      atomicAdd(reinterpret_cast<double*>(&p.stats[4]), ret);
    }
    if (p.done_count && sh_u[4]) atomicAdd(p.done_count, sh_u[4]);
  }
}

// ---- V consecutive envs: step, then (AUTO) same-step reset --------------------------------
// Phase 1 runs the branch-free dynamics of all V envs back to back (independent chains the
// scheduler can interleave); an env whose fast-path precondition fails is redone with the
// reference form.  Phase 2 serves the finished envs one per lane per pass: a lane with one
// finished env draws ONE Philox block, whichever of its V slots that env sits in, so a warp
// runs the reset code about once per step instead of once per slot.
template <int KIND, int V>
struct Group {
  using E = Env<KIND>;
  float st[V][E::SD];
  uint32_t steps[V], sbt[V];
  float ret[V];
  // per-step outputs
  float obs[V][E::OD], fin[V][E::OD], reward[V];
  uint32_t flags[V];
};

// What step_group does with the envs that finished (AUTO only):
//   RESET_IN_PLACE  tallies them and draws their reset states right away (per-call step, LDG form)
//   RESET_BY_CALLER neither tallies nor resets.  The rollout kernel does both behind ONE warp vote, so a step in
//                   which no env of the warp finished pays nothing for statistics or resets; the TMA step kernel
//                   tallies from the packed flags word and hands the finished envs to its reset warp.
enum ResetMode : int { RESET_IN_PLACE = 0, RESET_BY_CALLER = 2 };

// The reset state of an env is a function of (seed; global env index, step index at which the episode that just
// finished BEGAN): Philox counter (g, t_start).  The start index is known for the whole episode (t_start = t - count
// at the entry of step t), so -- unlike a stream keyed by the finishing step -- the state an env will restart
// from can be drawn at any time before it is needed: the rollout kernel draws it ahead of time with full warps.
__device__ __forceinline__ uint64_t episode_start(uint64_t t, uint32_t count_after) { return t + 1ull - (uint64_t)count_after; }

// Reset states drawn ahead of time (rollout kernel, kinds with Env::PREFETCH_RESETS): per thread one slot of shared
// memory per env, and a validity bit per slot.  A null `smem` means "none".
struct ResetPrefetch {
  float4* smem = nullptr;  // this thread's slot 0; slot v at smem[v * 256]
  uint32_t valid = 0;      // bit v: slot v holds the state for the END of env v's current episode
};

// The parameters of the new episodes of the slots in `pending` (p is a KernelParamsR), one slot per lane per pass,
// from Philox whatever the source of the reset state, stored to `rd`.  Runs right before reset_pending (it reads the
// counts AFTER the finishing step, which reset_pending clears).
template <int KIND, int V>
__device__ __forceinline__ void redraw_pending(const KernelParams& p, uint64_t base, uint64_t t, uint32_t pending,
                                               const Group<KIND, V>& g, const RedrawDst& rd) {
  const ParamBox& box = static_cast<const KernelParamsR&>(p).redraw;
  while (pending) {
    const int sel = __ffs(pending) - 1;
    pending &= pending - 1;
    uint32_t count = g.steps[0];
#pragma unroll
    for (int v = 1; v < V; ++v) count = (v == sel) ? g.steps[v] : count;
    redraw_params<Env<KIND>::NP>(p.keys, box, p.env_base + base + sel, episode_start(t, count), TAG_REDRAW_AUTO,
                                 rd.base + (uint64_t)sel * rd.vstride, rd.cstride);
  }
}

// Draws the reset states of the slots in `pending` (bit v = slot v), one slot per lane per pass.  g.steps[] are the
// counts AFTER the finishing step (they are cleared here).
template <int KIND, int V>
__device__ __forceinline__ void reset_pending(const KernelParams& p, uint64_t base, uint64_t t, uint32_t pending,
                                              Group<KIND, V>& g, ResetPrefetch* pre = nullptr) {
  using E = Env<KIND>;
  while (pending) {
    const int sel = __ffs(pending) - 1;
    pending &= pending - 1;
    const uint64_t gid = p.env_base + base + sel;
    uint32_t count = g.steps[0];
#pragma unroll
    for (int v = 1; v < V; ++v) count = (v == sel) ? g.steps[v] : count;
    float ns[E::SD], no[E::OD];
    if (p.reset_pool) {
      const uint64_t j = (gid + t) % p.pool_len;
#pragma unroll
      for (int c = 0; c < E::SD; ++c) ns[c] = p.reset_pool[(uint64_t)c * p.pool_len + j];
    } else if (pre) {  // the caller has redrawn every pending slot that was not valid
      const float4 q = pre->smem[sel * 256];
      const float qs[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int c = 0; c < E::SD && c < 4; ++c) ns[c] = qs[c];
    } else {
      E::reset(philox_env(p.keys, gid, episode_start(t, count), TAG_AUTO_RESET), ns);
    }
    if (pre) pre->valid &= ~(1u << sel);  // the new episode's own reset state has not been drawn yet
    if constexpr (!E::OBS_IS_STATE) E::obs(ns, no);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const bool hit = v == sel;
#pragma unroll
      for (int c = 0; c < E::SD; ++c) g.st[v][c] = hit ? ns[c] : g.st[v][c];
      if constexpr (!E::OBS_IS_STATE) {
#pragma unroll
        for (int c = 0; c < E::OD; ++c) g.obs[v][c] = hit ? no[c] : g.obs[v][c];
      }
      g.steps[v] = hit ? 0u : g.steps[v];
      g.ret[v] = hit ? 0.0f : g.ret[v];
    }
  }
}

// The flags of a group packed one byte per slot (what the flags store writes for V = 4).
template <int KIND, int V>
__device__ __forceinline__ uint32_t packed_flags(const Group<KIND, V>& g) {
  static_assert(V <= 4, "one byte per slot");
  uint32_t w = 0;
#pragma unroll
  for (int v = 0; v < V; ++v) w |= g.flags[v] << (8 * v);
  return w;
}

// Episode statistics of the finished slots from the packed flags: three population counts per group instead
// of three selects and adds per env.  Must run BEFORE reset_pending (it reads the finishing counters / returns).
template <int KIND, int V, bool TALLY_LEN>
__device__ __forceinline__ void tally_packed(uint32_t w, const Group<KIND, V>& g, StatAcc& acc) {
  using E = Env<KIND>;
  acc.episodes += __popc((w | (w >> 1)) & 0x01010101u);
  acc.terminated += __popc(w & 0x01010101u);
  acc.truncated += __popc(w & 0x02020202u);
  if constexpr (TALLY_LEN || !E::ANALYTIC_RETURN) {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const bool hit = ((w >> (8 * v)) & 0xffu) != 0;
      if constexpr (TALLY_LEN) acc.length_sum += hit ? g.steps[v] : 0u;
      if constexpr (!E::ANALYTIC_RETURN) {
        if (hit) acc.return_sum += (double)g.ret[v];
      }
    }
  }
}

// Do all V slots satisfy the kind's entry invariant (always true for kinds without one)?
template <int KIND, int V>
__device__ __forceinline__ bool group_trusted(const Group<KIND, V>& g) {
  bool mine = true;
  if constexpr (Env<KIND>::HAS_TRUSTED) {
#pragma unroll
    for (int v = 0; v < V; ++v) mine = mine && Env<KIND>::trusted_entry(g.st[v]);
  }
  return mine;
}

// The cold path of step_group: the reference form for every env of a lane that holds one outside the fast forms'
// precondition.  Out of line on purpose: inlined, its long sinf/cosf/fmodf reductions sit in the middle of the hot
// function and the register allocator pays for them on the hot path (Pendulum's step: +14 % instructions, mostly
// re-loaded constants); as a call it costs the hot path nothing.
// Arguments and results travel BY VALUE in one struct: a reference to the caller's own state array would make that
// array live in local memory on the hot path too.
template <int KIND, int V>
struct LaneIO {
  float st[V][Env<KIND>::SD];
  float aux[V];
  typename Env<KIND>::act_t action[V];
};
template <int KIND, int V>
__device__ __noinline__ LaneIO<KIND, V> dynamics_reference_lane(LaneIO<KIND, V> io, const EnvConsts& k) {
#pragma unroll 1
  for (int v = 0; v < V; ++v) Env<KIND>::dynamics(io.st[v], io.action[v], k, io.aux[v]);
  return io;
}

// TRUSTED (kinds with Env::HAS_TRUSTED): the caller has established Env::trusted_entry for every slot, which the
// dynamics themselves then preserve, so the fast form runs without its per-step precondition test.
// OBS_VALID (kinds with Env::HAS_OBS_CACHE): g.obs is the observation of the state in g.st on entry.
// PR (ParamRows with NP > 0): every env steps with its own constants, prm.r[.][v] (Env::dynamics_p).
// REDRAW (RESET_IN_PLACE, p is a KernelParamsR): the reset also redraws the finished envs' parameter rows in global
// memory (the step itself ran on the old ones, in prm).
template <int KIND, int V, bool AUTO, bool WANT_FINAL, bool TALLY_LEN = true, int RESET = RESET_IN_PLACE,
          bool TRUSTED = false, bool OBS_VALID = false, typename PR = NoParams, bool REDRAW = false>
__device__ __forceinline__ void step_group(const KernelParams& p, bool count, uint64_t base, uint64_t t,
                                           const typename Env<KIND>::act_t (&action)[V], bool track_ret,
                                           Group<KIND, V>& g, StatAcc& acc, const PR& prm = PR{}) {
  using E = Env<KIND>;
  float aux[V];
#pragma unroll
  for (int v = 0; v < V; ++v) aux[v] = 0.0f;
  if constexpr (PR::NP > 0) {
    static_assert(PR::NP == E::NP, "parameter rows of another kind");
    // Kinds whose fast form does not depend on the constants (PARAM_FAST) keep it, behind the same test of the
    // step's inputs as below; the others run the reference form with the env's constants.
    bool fast = false;
    if constexpr (E::PARAM_FAST) {
      fast = true;
      if constexpr (!(TRUSTED && E::HAS_TRUSTED)) {
#pragma unroll
        for (int v = 0; v < V; ++v) fast = fast & E::fast_ok(g.st[v], action[v], p.k);
      }
    }
    constexpr bool CACHED = OBS_VALID && E::HAS_OBS_CACHE;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float pe[E::NP];
#pragma unroll
      for (int c = 0; c < E::NP; ++c) pe[c] = prm.r[c][v];
      const float sin_cached = CACHED ? g.obs[v][E::OD > 1 ? 1 : 0] : 0.0f;
      if (fast)
        E::template dynamics_p<true, CACHED>(g.st[v], action[v], p.k, pe, aux[v], sin_cached);
      else
        E::template dynamics_p<false, false>(g.st[v], action[v], p.k, pe, aux[v], 0.0f);
    }
  } else if constexpr (E::HAS_BATCH) {
    // Acrobot: the RK4 stages test their own intermediates, so the fast form runs first (it writes the state
    // unconditionally) and an env whose test failed is restored from here and redone with the reference form
    bool ok[V];
    bool all_ok = true;
    float old[V][E::SD];
#pragma unroll
    for (int v = 0; v < V; ++v) {
#pragma unroll
      for (int c = 0; c < E::SD; ++c) old[v][c] = g.st[v][c];
    }
    E::template dynamics_fast_batch<V>(g.st, action, p.k, ok);
#pragma unroll
    for (int v = 0; v < V; ++v) all_ok = all_ok && ok[v];
    if (!all_ok) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        if (!ok[v]) {
#pragma unroll
          for (int c = 0; c < E::SD; ++c) g.st[v][c] = old[v][c];
          E::dynamics(g.st[v], action[v], p.k, aux[v]);
        }
      }
    }
  } else {
    // The precondition of the fast forms is a function of the inputs: test it first.  A lane that holds an env
    // outside it (rare: states nobody reaches by stepping) runs the reference form for all its envs -- the two
    // forms agree bit for bit wherever the fast one applies, so results do not depend on the path taken.
    bool all_ok = true;
    if constexpr (!(TRUSTED && E::HAS_TRUSTED)) {
#pragma unroll
      for (int v = 0; v < V; ++v) all_ok = all_ok & E::fast_ok(g.st[v], action[v], p.k);
      all_ok = all_ok & E::fast_enabled(p.k);
    }
    if (all_ok) {
      if constexpr (E::HAS_GROUP) {
        E::template dynamics_fast_group<V>(g.st, action, p.k);
      } else if constexpr (E::HAS_PAIR && V % 2 == 0) {
#pragma unroll
        for (int v = 0; v < V; v += 2) {
          bool oka, okb;
          E::dynamics_fast2(g.st[v], g.st[v + 1], action[v], action[v + 1], p.k, oka, okb);
        }
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          if constexpr (OBS_VALID && E::HAS_OBS_CACHE) {
            E::dynamics_fast_cached(g.st[v], action[v], p.k, aux[v], g.obs[v]);
          } else {
            E::dynamics_fast(g.st[v], action[v], p.k, aux[v]);
          }
        }
      }
    } else {
      LaneIO<KIND, V> io;
#pragma unroll
      for (int v = 0; v < V; ++v) {
#pragma unroll
        for (int c = 0; c < E::SD; ++c) io.st[v][c] = g.st[v][c];
        io.aux[v] = 0.0f;
        io.action[v] = action[v];
      }
      io = dynamics_reference_lane<KIND, V>(io, p.k);
#pragma unroll
      for (int v = 0; v < V; ++v) {
#pragma unroll
        for (int c = 0; c < E::SD; ++c) g.st[v][c] = io.st[v][c];
        aux[v] = io.aux[v];
      }
    }
  }
  uint32_t pending = 0;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    if constexpr (AUTO) g.sbt[v] = SBT_NONE;  // auto-reset presumes reset() precedes every episode
    if constexpr (E::OUTCOME_FROM_OBS) {
      E::obs(g.st[v], g.obs[v]);
      g.flags[v] = E::template outcome_obs<!AUTO>(g.st[v], g.obs[v], g.steps[v], p.k, g.reward[v]);
    } else {
      g.flags[v] = E::template outcome<!AUTO>(g.st[v], action[v], aux[v], g.steps[v], g.sbt[v], p.k, g.reward[v]);
    }
    if (track_ret) g.ret[v] = fadd(g.ret[v], g.reward[v]);
    if constexpr (!E::OBS_IS_STATE || WANT_FINAL) {
      if constexpr (!E::OUTCOME_FROM_OBS) E::obs(g.st[v], g.obs[v]);
      if constexpr (WANT_FINAL) {
#pragma unroll
        for (int c = 0; c < E::OD; ++c) g.fin[v][c] = g.obs[v][c];
      }
    }
    if constexpr (AUTO && RESET != RESET_BY_CALLER) {
      const bool done = g.flags[v] != 0;
      pending |= done ? (1u << v) : 0u;
      // flags are 0 for a live env, so the masks need no extra select
      const uint32_t fl = count ? g.flags[v] : 0u;
      acc.episodes += fl != 0 ? 1u : 0u;
      acc.terminated += fl & FLAG_TERMINATED;
      acc.truncated += fl >> 1;
      if constexpr (TALLY_LEN) acc.length_sum += fl != 0 ? g.steps[v] : 0u;
      const bool tally = fl != 0;
      if constexpr (!E::ANALYTIC_RETURN) {
        if (tally) acc.return_sum += (double)g.ret[v];
      }
    }
  }
  if constexpr (AUTO && RESET == RESET_IN_PLACE && REDRAW) {
    const RedrawDst rd{const_cast<float*>(static_cast<const KernelParamsP&>(p).params) + base, p.ld, 1};
    redraw_pending<KIND, V>(p, base, t, pending, g, rd);
  }
  if constexpr (AUTO && RESET == RESET_IN_PLACE) reset_pending<KIND, V>(p, base, t, pending, g);
}

template <int MODE>
struct CounterType {
  using type = uint32_t;
};
template <>
struct CounterType<CNT_S16> {
  using type = uint16_t;
};
// stored value -> episode step count at the entry of step t, and back (t_next = the step index the count belongs to)
template <int CNT>
__device__ __forceinline__ uint32_t cnt_decode(typename CounterType<CNT>::type raw, uint64_t t) {
  using cnt_t = typename CounterType<CNT>::type;
  if constexpr (cnt_is_stamp(CNT)) return (uint32_t)(cnt_t)((uint32_t)t - (uint32_t)raw);
  return raw;
}
template <int CNT>
__device__ __forceinline__ typename CounterType<CNT>::type cnt_encode(uint32_t steps, uint64_t t_next) {
  using cnt_t = typename CounterType<CNT>::type;
  if constexpr (cnt_is_stamp(CNT)) return (cnt_t)((uint32_t)t_next - steps);
  return (cnt_t)steps;
}

// =============================================================================================
// Mode 1: per-call step kernel
// =============================================================================================
// REDRAW: every reset also redraws the env's parameter rows (mgym_set_param_redraw; auto-reset with rows only).
template <int KIND, int V, bool AUTO, int CNT, bool PARAMS = false, bool REDRAW = false>
__global__ void __launch_bounds__(256, 1) step_kernel(const __grid_constant__ KParams<PARAMS, REDRAW> p) {
  using E = Env<KIND>;
  using act_t = typename E::act_t;
  using cnt_t = typename CounterType<CNT>::type;
  using PR = ParamRows<PARAMS ? E::NP : 0, V>;
  constexpr int SD = E::SD, OD = E::OD;
  static_assert(!REDRAW || (PARAMS && AUTO), "redraw is a form of the auto-reset parameter kernels");
  static_assert(!cnt_is_lazy(CNT) && (AUTO || !cnt_is_stamp(CNT)), "the host maps CNT_S32_LAZY to CNT_S32 here");
  StatAcc acc;
  const uint64_t groups = p.n / V;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const bool track_ret = !E::ANALYTIC_RETURN && p.ep_return != nullptr;
  const bool want_final = p.final_obs_out != nullptr;
  const uint64_t t_now = launch_t(p);

  for (uint64_t grp = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; grp < groups; grp += stride) {
    const uint64_t base = p.first + grp * V;
    Group<KIND, V> g;
    act_t action[V];
    PR prm;
    if constexpr (PARAMS) {
#pragma unroll
      for (int c = 0; c < E::NP; ++c) {
        const Vec<float, V> r = ldv<float, V>(p.params + (uint64_t)c * p.ld + base);
#pragma unroll
        for (int v = 0; v < V; ++v) prm.r[c][v] = r.v[v];
      }
    }
    {
      Vec<float, V> s[SD];
#pragma unroll
      for (int c = 0; c < SD; ++c) s[c] = ldv<float, V>(p.state + (uint64_t)c * p.ld + base);
      const Vec<act_t, V> a = ldv<act_t, V>(reinterpret_cast<const act_t*>(p.actions) + base);
      const Vec<cnt_t, V> cnt = ldv<cnt_t, V>(reinterpret_cast<const cnt_t*>(p.steps) + base);
      Vec<uint32_t, V> sb;
      if constexpr (!AUTO && KIND == 0) sb = ldv<uint32_t, V>(p.sbt + base);
      Vec<float, V> er;
      if (track_ret) er = ldv<float, V>(p.ep_return + base);
#pragma unroll
      for (int v = 0; v < V; ++v) {
#pragma unroll
        for (int c = 0; c < SD; ++c) g.st[v][c] = s[c].v[v];
        action[v] = a.v[v];
        g.steps[v] = cnt_decode<CNT>(cnt.v[v], t_now);
        g.sbt[v] = SBT_NONE;
        if constexpr (!AUTO && KIND == 0) g.sbt[v] = sb.v[v];
        g.ret[v] = track_ret ? er.v[v] : 0.0f;
      }
    }
    if (want_final)
      step_group<KIND, V, AUTO, true, true, RESET_IN_PLACE, false, false, PR, REDRAW>(p, true, base, t_now, action, track_ret,
                                                                                     g, acc, prm);
    else
      step_group<KIND, V, AUTO, false, true, RESET_IN_PLACE, false, false, PR, REDRAW>(p, true, base, t_now, action, track_ret,
                                                                                      g, acc, prm);

    {
      Vec<float, V> s[SD];
#pragma unroll
      for (int c = 0; c < SD; ++c) {
#pragma unroll
        for (int v = 0; v < V; ++v) s[c].v[v] = g.st[v][c];
        stv<float, V>(p.state + (uint64_t)c * p.ld + base, s[c]);
      }
    }
    // a start stamp only changes when an episode ended (the count of a finished env is 0 again by now)
    if (!cnt_is_stamp(CNT) || packed_flags<KIND, V>(g) != 0u) {
      Vec<cnt_t, V> cnt;
#pragma unroll
      for (int v = 0; v < V; ++v) cnt.v[v] = cnt_encode<CNT>(g.steps[v], t_now + 1);
      stv<cnt_t, V>(reinterpret_cast<cnt_t*>(p.steps) + base, cnt);
    }
    if constexpr (!AUTO && KIND == 0) {
      Vec<uint32_t, V> sb;
#pragma unroll
      for (int v = 0; v < V; ++v) sb.v[v] = g.sbt[v];
      stv<uint32_t, V>(p.sbt + base, sb);
    }
    if (track_ret) {
      Vec<float, V> er;
#pragma unroll
      for (int v = 0; v < V; ++v) er.v[v] = g.ret[v];
      stv<float, V>(p.ep_return + base, er);
    }
    if (p.obs_out) {
#pragma unroll
      for (int c = 0; c < OD; ++c) {
        Vec<float, V> o;
#pragma unroll
        for (int v = 0; v < V; ++v) o.v[v] = E::OBS_IS_STATE ? g.st[v][c < SD ? c : 0] : g.obs[v][c];
        stv<float, V>(p.obs_out + (uint64_t)c * p.ld + base, o);
      }
    }
    if (want_final) {
#pragma unroll
      for (int c = 0; c < OD; ++c) {
        Vec<float, V> o;
#pragma unroll
        for (int v = 0; v < V; ++v) o.v[v] = g.fin[v][c];
        stv<float, V>(p.final_obs_out + (uint64_t)c * p.ld + base, o);
      }
    }
    if (p.reward_out) {
      Vec<float, V> rw;
#pragma unroll
      for (int v = 0; v < V; ++v) rw.v[v] = g.reward[v];
      stv<float, V>(p.reward_out + base, rw);
    }
    if (p.flags_out) {
      Vec<uint8_t, V> fl;
#pragma unroll
      for (int v = 0; v < V; ++v) fl.v[v] = (uint8_t)g.flags[v];
      stv<uint8_t, V>(p.flags_out + base, fl);
    }
  }
  if constexpr (AUTO) stats_flush<KIND>(acc, p);
  fused_clock_advance(p);
}

// =============================================================================================
// Mode 1, TMA-staged: the same step, with the inputs of each warp's next tiles already in flight.
//
// The LDG form above can only keep (resident warps x 76 B x 32 lanes) of reads in flight, and the
// register budget of the interleaved 4-env arithmetic caps resident warps at 16-32 per SM -- not
// enough bytes in flight to cover HBM latency (ncu: long-scoreboard stalls at the loads, DRAM < 50 %).
// Here every CTA owns a ring of STAGES shared-memory tiles (1024 envs each: SD state rows, actions,
// counters, ~19 KB) that a dedicated producer warp fills with cp.async.bulk (TMA, 1-D bulk copies
// completing on an mbarrier).  Bytes in flight no longer depend on occupancy: CTAs x STAGES x 19 KB.
// =============================================================================================
namespace tma {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
}  // namespace tma

constexpr int TMA_STAGES = 4;
constexpr int TMA_CONSUMER_WARPS = 8;
constexpr int TMA_THREADS = (TMA_CONSUMER_WARPS + 2) * 32;  // + one producer warp + one reset warp
constexpr int TMA_RESET_BUFFERS = 2;                         // request queues in flight
constexpr int TMA_TILE = TMA_CONSUMER_WARPS * 32 * 4;       // envs per CTA tile: 256 consumer threads x V=4

// PARAMS: the env's NP parameter rows travel with the tile (4 NP bytes per env more).  The stage count is then the
// largest (up to TMA_STAGES) that still lets two CTAs share an SM: CartPole's 43 KB stage runs 2 stages x 2 CTAs
// (4 tiles = 172 KB in flight per SM, against 4 x 2 x 19 KB without parameters).
template <int KIND, int CNT, bool AUTO = true, bool PARAMS = false>
struct TmaLayout {
  using E = Env<KIND>;
  static constexpr uint32_t ROW = TMA_TILE * 4;  // one f32 row of a tile
  static constexpr uint32_t OFF_ACT = E::SD * ROW;
  static constexpr uint32_t ACT_BYTES = TMA_TILE * sizeof(typename E::act_t);
  static constexpr uint32_t OFF_CNT = OFF_ACT + ACT_BYTES;
  static constexpr uint32_t CNT_BYTES = cnt_staged(CNT) ? TMA_TILE * sizeof(typename CounterType<CNT>::type) : 0;
  static constexpr uint32_t OFF_RET = OFF_CNT + CNT_BYTES;
  static constexpr uint32_t RET_BYTES = (E::ANALYTIC_RETURN || !AUTO) ? 0 : ROW;
  // manual CartPole also carries steps_beyond_terminated (cartpole.rs:27)
  static constexpr uint32_t OFF_SBT = OFF_RET + RET_BYTES;
  static constexpr uint32_t SBT_BYTES = (!AUTO && KIND == 0) ? ROW : 0;
  static constexpr uint32_t OFF_PAR = OFF_SBT + SBT_BYTES;
  static constexpr uint32_t PAR_BYTES = PARAMS ? E::NP * ROW : 0;
  static constexpr uint32_t STAGE_BYTES = (OFF_PAR + PAR_BYTES + 127u) & ~127u;
  static constexpr uint32_t BAR_BYTES = 128;  // full[STAGES], empty[STAGES], tile id of each stage
  static_assert(24 * TMA_STAGES <= 128, "barriers and tile ids must fit BAR_BYTES");
  // reset queues: per buffer {q_full, q_empty mbarriers, tile id, count} (32 B) + per finished env its uint16 index in
  // the tile and the uint32 length of the episode that ended (the reset stream is keyed by its start)
  static constexpr uint32_t QUEUE_STRIDE = 32 + TMA_TILE * 2 + TMA_TILE * 4;
  static constexpr uint32_t QUEUE_BYTES = TMA_RESET_BUFFERS * QUEUE_STRIDE;
  static constexpr int fit_stages() {
    const uint32_t budget = 110u * 1024u - 256u - QUEUE_BYTES;  // per CTA, two CTAs per SM
    const int s = (int)(budget / STAGE_BYTES);
    return s > TMA_STAGES ? TMA_STAGES : (s < 1 ? 1 : s);
  }
  static constexpr int STAGES = PARAMS ? fit_stages() : TMA_STAGES;
  static constexpr uint32_t OFF_QUEUE = BAR_BYTES + STAGES * STAGE_BYTES;
  static constexpr uint32_t SMEM_BYTES = 128 + OFF_QUEUE + QUEUE_BYTES;
};

// Warp-specialised: warp 8 is the TMA producer (one elected lane draws a tile ticket, arms full[s] and
// launches the six bulk copies of a 1024-env tile once the consumers have released stage s through
// empty[s]); warps 0-7 are consumers (wait full[s], pull their 4 envs out of shared memory, release the
// stage, step, store straight from registers); warp 9 is the reset warp.
//
// Reset warp.  A finished env needs a Philox block and four f64->f32 uniforms (~130 instructions), but only
// 4-6 lanes of a consumer warp have one per step, so done in place that costs every consumer warp a whole
// pass: ~25 % of all issued instructions, and under the 1 kW power cap the step is issue-bound.  Instead the
// consumers only APPEND the finished env's index to a shared-memory queue (and clear its counter), store the
// tile, and arrive on q_full[b] -- whose release orders their stores before whatever the reset warp does
// next.  The reset warp then draws the new states with all 32 lanes busy (46 per tile on average = 2
// passes per 1024 envs instead of 10) and patches them into the state rows (and obs_out) in global memory.
// Consumers never wait for it except to reuse a queue buffer two tiles later.
//
// AUTO = false is the reference's own protocol (no same-step reset: the caller resets what finished,
// cartpole.rs:468-470): the same pipeline with steps_beyond_terminated as one more row and nothing ever queued
// for the reset warp.
//
// REDRAW (mgym_set_param_redraw): the reset warp also draws the new episode's parameters of each queued env (one more
// Philox block, two for CartPole) and writes them into the rows in global memory.  The consumers stepped that tile
// with the staged (old) rows; no other tile of the launch holds the env, and the next launch's producer reads the
// rows only after griddepcontrol.wait.  Stage layout and stage count are those of the PARAMS form.
template <int KIND, int CNT, bool AUTO = true, bool PARAMS = false, bool REDRAW = false>
__global__ void __launch_bounds__(TMA_THREADS, 2)
    step_kernel_tma(const __grid_constant__ KParams<PARAMS, REDRAW> p) {
  using E = Env<KIND>;
  using L = TmaLayout<KIND, CNT, AUTO, PARAMS>;
  using act_t = typename E::act_t;
  using cnt_t = typename CounterType<CNT>::type;
  constexpr int SD = E::SD, OD = E::OD, V = 4;
  constexpr int TMA_STAGES = L::STAGES;  // shadows the global default: this kernel's own ring depth
  using PR = ParamRows<PARAMS ? E::NP : 0, V>;
  static_assert(!REDRAW || (PARAMS && AUTO), "redraw is a form of the auto-reset parameter kernels");
  static_assert(AUTO || !cnt_is_stamp(CNT), "manual mode keeps the reference's own counters");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (tma::smem_u32(smem_raw) + 127u) & ~127u;
  const uint32_t warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // warp-uniform for the compiler
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t full0 = smem_base, empty0 = smem_base + 8 * TMA_STAGES;
  volatile uint64_t* tile_slot =
      reinterpret_cast<volatile uint64_t*>(smem_raw + (smem_base + 16 * TMA_STAGES - tma::smem_u32(smem_raw)));
  // reset queues, one per buffer: [q_full mbarrier][q_empty mbarrier][tile id u64][count u32, pad][uint16 x TMA_TILE]
  // [uint32 x TMA_TILE]
  constexpr uint32_t QSTRIDE = L::QUEUE_STRIDE;
  const uint32_t queue0 = smem_base + L::OFF_QUEUE;
  uint8_t* const queue_ptr = smem_raw + (queue0 - tma::smem_u32(smem_raw));
  auto q_tile = [&](uint32_t b) { return reinterpret_cast<volatile uint64_t*>(queue_ptr + b * QSTRIDE + 16); };
  auto q_count = [&](uint32_t b) { return reinterpret_cast<uint32_t*>(queue_ptr + b * QSTRIDE + 24); };
  auto q_items = [&](uint32_t b) { return reinterpret_cast<uint16_t*>(queue_ptr + b * QSTRIDE + 32); };
  auto q_lengths = [&](uint32_t b) { return reinterpret_cast<uint32_t*>(queue_ptr + b * QSTRIDE + 32 + TMA_TILE * 2); };
  const uint32_t data0 = smem_base + L::BAR_BYTES;
  const uint64_t n_tiles = p.n / TMA_TILE;
  const bool track_ret = AUTO && !E::ANALYTIC_RETURN && p.ep_return != nullptr;
  const bool want_final = p.final_obs_out != nullptr;
  constexpr bool HAS_SBT = !AUTO && KIND == 0;
  StatAcc acc;

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < TMA_STAGES; ++s) {
      tma::mbar_init(full0 + 8 * s, 1);
      tma::mbar_init(empty0 + 8 * s, TMA_CONSUMER_WARPS);
    }
    for (int b = 0; b < TMA_RESET_BUFFERS; ++b) {
      tma::mbar_init(queue0 + b * QSTRIDE, TMA_CONSUMER_WARPS);  // q_full: every consumer warp has stored its tile
      tma::mbar_init(queue0 + b * QSTRIDE + 8, 1);               // q_empty: the reset warp is done with the buffer
      *q_count(b) = 0u;
    }
    tma::fence_mbar_init();
  }
  __syncthreads();
  // Programmatic dependent launch: everything above overlaps the tail of the previous launch on this
  // stream (usually the previous step); nothing below may run before that launch has completed and
  // flushed.  Our own dependents may start their prologue as soon as they find room.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;");
  const uint64_t t_now = launch_t(p), work_base = launch_work_base(p);  // only after the wait: see t_dev

  if (warp == TMA_CONSUMER_WARPS) {
    // ---------------- producer ----------------
    // Tiles are handed out by a global ticket counter (first come, first served), so CTAs that run faster
    // take more tiles and the launch ends with every CTA busy until the tickets run out.  Launch L owns the
    // tickets [work_base, work_base + n_tiles + gridDim.x): each CTA draws exactly one ticket past the end.
    if (lane == 0) {
      const act_t* actions = reinterpret_cast<const act_t*>(p.actions);
      const uint32_t tx =
          SD * L::ROW + L::ACT_BYTES + L::CNT_BYTES + (track_ret ? L::ROW : 0u) + L::SBT_BYTES + L::PAR_BYTES;
      for (uint32_t it = 0;; ++it) {
        const uint32_t s = it % TMA_STAGES, round = it / TMA_STAGES;
        tma::mbar_wait(empty0 + 8 * s, (round & 1u) ^ 1u);  // first round passes at once
        const uint64_t tile = atomicAdd(p.work_counter, 1ull) - work_base;
        const uint32_t bar = full0 + 8 * s, dst = data0 + s * L::STAGE_BYTES;
        tile_slot[s] = tile;
        if (tile >= n_tiles) {  // out of work: tell the consumers and stop
          tma::mbar_arrive(bar);
          break;
        }
        const uint64_t e0 = p.first + tile * TMA_TILE;
        tma::mbar_expect_tx(bar, tx);
#pragma unroll
        for (int c = 0; c < SD; ++c) tma::bulk_g2s(dst + c * L::ROW, p.state + (uint64_t)c * p.ld + e0, L::ROW, bar);
        tma::bulk_g2s(dst + L::OFF_ACT, actions + e0, L::ACT_BYTES, bar);
        if constexpr (cnt_staged(CNT))
          tma::bulk_g2s(dst + L::OFF_CNT, reinterpret_cast<const cnt_t*>(p.steps) + e0, L::CNT_BYTES, bar);
        if constexpr (!E::ANALYTIC_RETURN && AUTO) {
          if (track_ret) tma::bulk_g2s(dst + L::OFF_RET, p.ep_return + e0, L::ROW, bar);
        }
        if constexpr (HAS_SBT) tma::bulk_g2s(dst + L::OFF_SBT, p.sbt + e0, L::ROW, bar);
        if constexpr (PARAMS) {
#pragma unroll
          for (int c = 0; c < E::NP; ++c)
            tma::bulk_g2s(dst + L::OFF_PAR + c * L::ROW, p.params + (uint64_t)c * p.ld + e0, L::ROW, bar);
        }
      }
    }
    __syncwarp();
  } else if (warp == TMA_CONSUMER_WARPS + 1) {
    // ---------------- reset warp ----------------
    for (uint32_t it = 0;; ++it) {
      const uint32_t qb = it % TMA_RESET_BUFFERS, qround = it / TMA_RESET_BUFFERS;
      const uint32_t q_full = queue0 + qb * QSTRIDE, q_empty = q_full + 8;
      tma::mbar_wait(q_full, qround & 1u);  // acquire: every consumer warp's stores of this tile are visible
      const uint64_t tile = *q_tile(qb);
      if (tile >= n_tiles) break;
      const uint32_t count = *q_count(qb);
      const uint16_t* items = q_items(qb);
      const uint32_t* lengths = q_lengths(qb);
      const uint64_t tile_base = p.first + tile * TMA_TILE;
      for (uint32_t j = lane; j < count; j += 32) {
        const uint64_t local = tile_base + items[j];
        const uint64_t gid = p.env_base + local;
        float ns[SD];
        if (p.reset_pool) {
          const uint64_t k = (gid + t_now) % p.pool_len;
#pragma unroll
          for (int c = 0; c < SD; ++c) ns[c] = p.reset_pool[(uint64_t)c * p.pool_len + k];
        } else {
          E::reset(philox_env(p.keys, gid, episode_start(t_now, lengths[j]), TAG_AUTO_RESET), ns);
        }
        if constexpr (REDRAW) {
          redraw_params<E::NP>(p.keys, p.redraw, gid, episode_start(t_now, lengths[j]), TAG_REDRAW_AUTO,
                               const_cast<float*>(p.params) + local, p.ld);
        }
#pragma unroll
        for (int c = 0; c < SD; ++c) p.state[(uint64_t)c * p.ld + local] = ns[c];
        if (p.obs_out) {  // the observation the caller sees is the post-reset one
          float no[OD];
          E::obs(ns, no);
#pragma unroll
          for (int c = 0; c < OD; ++c) p.obs_out[(uint64_t)c * p.ld + local] = no[c];
        }
      }
      __syncwarp();
      if (lane == 0) {
        *q_count(qb) = 0u;
        tma::mbar_arrive(q_empty);
      }
    }
    __syncwarp();
  } else {
    // ---------------- consumers ----------------
    const uint32_t tid = threadIdx.x;  // 0..255
    for (uint32_t it = 0;; ++it) {
      const uint32_t s = it % TMA_STAGES, parity = (it / TMA_STAGES) & 1u;
      tma::mbar_wait(full0 + 8 * s, parity);
      const uint64_t tile = tile_slot[s];
      const uint32_t qb = it % TMA_RESET_BUFFERS, qround = it / TMA_RESET_BUFFERS;
      const uint32_t q_full = queue0 + qb * QSTRIDE, q_empty = q_full + 8;
      tma::mbar_wait(q_empty, (qround & 1u) ^ 1u);  // the reset warp has finished this buffer's previous tile
      if (tid == 0) *q_tile(qb) = tile;              // also carries the end-of-work sentinel
      if (tile >= n_tiles) {
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(q_full);
        break;
      }
      const uint64_t base = p.first + tile * TMA_TILE + tid * V;

      Group<KIND, V> g;
      act_t action[V];
      PR prm;
      {
        const uint8_t* st = smem_raw + (data0 + s * L::STAGE_BYTES - tma::smem_u32(smem_raw));
        if constexpr (PARAMS) {
#pragma unroll
          for (int c = 0; c < E::NP; ++c) {
            const Vec<float, V> r = ldv<float, V>(reinterpret_cast<const float*>(st + L::OFF_PAR + c * L::ROW) + tid * V);
#pragma unroll
            for (int v = 0; v < V; ++v) prm.r[c][v] = r.v[v];
          }
        }
        Vec<float, V> row[SD];
#pragma unroll
        for (int c = 0; c < SD; ++c) row[c] = ldv<float, V>(reinterpret_cast<const float*>(st + c * L::ROW) + tid * V);
        const Vec<act_t, V> a = ldv<act_t, V>(reinterpret_cast<const act_t*>(st + L::OFF_ACT) + tid * V);
        Vec<cnt_t, V> cnt;
        if constexpr (cnt_staged(CNT)) cnt = ldv<cnt_t, V>(reinterpret_cast<const cnt_t*>(st + L::OFF_CNT) + tid * V);
        Vec<float, V> er;
        if constexpr (!E::ANALYTIC_RETURN && AUTO) {
          if (track_ret) er = ldv<float, V>(reinterpret_cast<const float*>(st + L::OFF_RET) + tid * V);
        }
        Vec<uint32_t, V> sb;
        if constexpr (HAS_SBT) sb = ldv<uint32_t, V>(reinterpret_cast<const uint32_t*>(st + L::OFF_SBT) + tid * V);
#pragma unroll
        for (int v = 0; v < V; ++v) {
#pragma unroll
          for (int c = 0; c < SD; ++c) g.st[v][c] = row[c].v[v];
          action[v] = a.v[v];
          g.steps[v] = 0;
          g.sbt[v] = SBT_NONE;
          if constexpr (cnt_staged(CNT)) g.steps[v] = cnt_decode<CNT>(cnt.v[v], t_now);
          if constexpr (HAS_SBT) g.sbt[v] = sb.v[v];
          g.ret[v] = 0.0f;
          if constexpr (!E::ANALYTIC_RETURN && AUTO) g.ret[v] = track_ret ? er.v[v] : 0.0f;
        }
      }
      __syncwarp();  // every lane of this warp has its values in registers
      if (lane == 0) tma::mbar_arrive(empty0 + 8 * s);

      if (want_final)
        step_group<KIND, V, AUTO, true, true, RESET_BY_CALLER, false, false, PR>(p, true, base, t_now, action, track_ret,
                                                                                  g, acc, prm);
      else
        step_group<KIND, V, AUTO, false, true, RESET_BY_CALLER, false, false, PR>(p, true, base, t_now, action, track_ret,
                                                                                   g, acc, prm);
      // Everything about this lane's finished envs sits in one branch: statistics from the packed flags word,
      // counters cleared, and their index inside the tile appended to the reset queue.
      const uint32_t fw = packed_flags<KIND, V>(g);
      // in manual mode finished envs wait for the caller's reset
      const uint32_t fin = AUTO ? fw : 0u;
      if (fin) {
        if constexpr (cnt_is_lazy(CNT)) {
          // the episode length is only needed now: the stamps of this lane's envs come straight from global memory
          const Vec<cnt_t, V> sv = ldv<cnt_t, V>(reinterpret_cast<const cnt_t*>(p.steps) + base);
#pragma unroll
          for (int v = 0; v < V; ++v) g.steps[v] = cnt_decode<CNT>(sv.v[v], t_now) + 1u;
        }
        tally_packed<KIND, V, true>(fin, g, acc);
        uint32_t pos = atomicAdd(q_count(qb), (uint32_t)__popc((fin | (fin >> 1)) & 0x01010101u));
        uint16_t* items = q_items(qb);
        uint32_t* lengths = q_lengths(qb);
#pragma unroll
        for (int v = 0; v < V; ++v) {
          if ((fin >> (8 * v)) & 0xffu) {
            items[pos] = (uint16_t)(tid * V + v);
            lengths[pos++] = g.steps[v];
            g.steps[v] = 0u;
            g.ret[v] = 0.0f;
          }
        }
        if constexpr (cnt_is_stamp(CNT)) {
          // new start stamps for the finished envs (the others re-encode to the value they had)
          Vec<cnt_t, V> sv;
#pragma unroll
          for (int v = 0; v < V; ++v) sv.v[v] = cnt_encode<CNT>(g.steps[v], t_now + 1);
          stv<cnt_t, V>(reinterpret_cast<cnt_t*>(p.steps) + base, sv);
        }
      }

#pragma unroll
      for (int c = 0; c < SD; ++c) {
        Vec<float, V> o;
#pragma unroll
        for (int v = 0; v < V; ++v) o.v[v] = g.st[v][c];
        stv<float, V>(p.state + (uint64_t)c * p.ld + base, o);
      }
      if constexpr (!cnt_is_stamp(CNT)) {
        Vec<cnt_t, V> cnt;
#pragma unroll
        for (int v = 0; v < V; ++v) cnt.v[v] = (cnt_t)g.steps[v];
        stv<cnt_t, V>(reinterpret_cast<cnt_t*>(p.steps) + base, cnt);
      }
      if constexpr (!E::ANALYTIC_RETURN && AUTO) {
        if (track_ret) {
          Vec<float, V> er;
#pragma unroll
          for (int v = 0; v < V; ++v) er.v[v] = g.ret[v];
          stv<float, V>(p.ep_return + base, er);
        }
      }
      if constexpr (HAS_SBT) {
        Vec<uint32_t, V> sbo;
#pragma unroll
        for (int v = 0; v < V; ++v) sbo.v[v] = g.sbt[v];
        stv<uint32_t, V>(p.sbt + base, sbo);
      }
      if (p.obs_out) {
#pragma unroll
        for (int c = 0; c < OD; ++c) {
          Vec<float, V> o;
#pragma unroll
          for (int v = 0; v < V; ++v) o.v[v] = E::OBS_IS_STATE ? g.st[v][c < SD ? c : 0] : g.obs[v][c];
          stv<float, V>(p.obs_out + (uint64_t)c * p.ld + base, o);
        }
      }
      if (want_final) {
#pragma unroll
        for (int c = 0; c < OD; ++c) {
          Vec<float, V> o;
#pragma unroll
          for (int v = 0; v < V; ++v) o.v[v] = g.fin[v][c];
          stv<float, V>(p.final_obs_out + (uint64_t)c * p.ld + base, o);
        }
      }
      if (p.reward_out) {
        Vec<float, V> rw;
#pragma unroll
        for (int v = 0; v < V; ++v) rw.v[v] = g.reward[v];
        stv<float, V>(p.reward_out + base, rw);
      }
      if (p.flags_out) *reinterpret_cast<uint32_t*>(p.flags_out + base) = fw;
      __syncwarp();
      if (lane == 0) tma::mbar_arrive(q_full);
    }
  }
  if constexpr (AUTO) stats_flush<KIND>(acc, p);
  fused_clock_advance(p);
}

// =============================================================================================
// Mode 2: fused K-step rollout kernel
// =============================================================================================
// FULL (chosen by the host): every warp tile is complete (n % (32 V) == 0), all three trajectory outputs are
// present and action validation is off -- the loop then carries no per-lane `active` predicate and no null
// tests.  Per step, everything that concerns finished envs (statistics, done count, Philox resets) sits behind
// ONE warp vote on the packed flags word: a warp tile in which nothing finished (MountainCar: almost always)
// pays one compare and one VOTE for it.
// Resident CTAs per SM the rollout is compiled for.  The loop is latency-bound at 16 warps per SM, and four of
// the kinds fit 80 registers without spilling (measured: +8..11 % at 3 CTAs); Acrobot's RK4 does not (-6 %).
template <int KIND>
constexpr int rollout_min_blocks() {
  return KIND == 4 ? 2 : 3;
}

// PARAMS: the NP parameters of each env are read once per warp tile into per-thread shared-memory slots (like the
// prefetched reset states) and picked up by every step: held in registers across the loop they would cost the
// occupancy the loop is built for.  The action ring is half as deep then, so that CartPole's slots (24 KB), its
// prefetched resets (16 KB) and the ring stay within the 48 KB of static shared memory.
// REDRAW (mgym_set_param_redraw): a reset also draws the finished env's parameters for its new episode, in the
// divergent reset pass, straight into its slots (every later step of the tile runs the new episode's constants); the
// slots are written back to the rows at the end of the tile.  Drawing them ahead of time like the reset states would
// need 24 KB more of CartPole's slots, i.e. dynamic shared memory (DESIGN.md section 11.1).
// FINAL (mgym_rollout_final, auto-reset forms only): the divergent reset pass also stores the observation each
// finished env ended on, before the reset overwrites it, to p.final_obs_out [K][OD][ld].  Only finished envs are
// written; the address is computed there from (kk, base), so the hot loop carries no extra pointer.
template <int KIND, int V, bool AUTO, int CNT, bool FULL, bool PARAMS = false, bool REDRAW = false, bool FINAL = false>
__global__ void __launch_bounds__(256, rollout_min_blocks<KIND>())
    rollout_kernel(const __grid_constant__ KParams<PARAMS, REDRAW> p) {
  using E = Env<KIND>;
  using act_t = typename E::act_t;
  using cnt_t = typename CounterType<CNT>::type;
  using PR = ParamRows<PARAMS ? E::NP : 0, V>;
  constexpr int SD = E::SD, OD = E::OD;
  static_assert(!REDRAW || (PARAMS && AUTO), "redraw is a form of the auto-reset parameter kernels");
  static_assert(!FULL || (AUTO && V == 4), "the FULL form is built for the vector auto-reset path only");
  static_assert(!FINAL || AUTO, "final observations exist only where the rollout resets");
  static_assert(!cnt_is_lazy(CNT) && (AUTO || !cnt_is_stamp(CNT)), "the host maps CNT_S32_LAZY to CNT_S32 here");
  constexpr int ACT_RING = PARAMS ? 4 : 8;  // steps of action look-ahead staged in shared memory
  __shared__ float par_slots[PARAMS ? E::NP * V : 1][PARAMS ? 256 : 1];  // [c * V + v][thread]
  static_assert((ACT_RING & (ACT_RING - 1)) == 0, "power of two");
  constexpr uint32_t RING_STRIDE = 256 * V * sizeof(act_t);  // one row of the CTA: 256 threads x V actions
  __shared__ __align__(16) act_t act_ring[V == 4 ? ACT_RING : 1][256 * V];
  // CartPole finishes an env every ~22 steps: ~6 of a warp's 128 envs per step, served by a divergent pass whose
  // Philox block + four f64 -> f32 uniforms run at ~6 of 32 lanes -- a third of all issued instructions.  The reset
  // stream is keyed by the START of the finished episode (reset_pending), so the state an env will restart from is
  // drawn AHEAD of time with all 32 lanes busy, into per-thread shared memory, and the divergent pass only picks it
  // up.  A slot is (re)drawn for the whole warp when some lane is about to consume it without a valid state (one
  // REDUX per step decides): every ~10 steps per slot in steady state, since an env must finish twice in between.
  constexpr bool PREFETCH = AUTO && V == 4 && E::PREFETCH_RESETS;
  __shared__ float4 next_reset[PREFETCH ? 4 : 1][256];
  StatAcc acc;
  uint32_t dones = 0;  // finished env-steps of this lane's groups
  const uint64_t groups = p.n / V;
  const bool track_ret = !E::ANALYTIC_RETURN && p.ep_return != nullptr;
  const bool policy = p.actions == nullptr;
  const act_t* actions = reinterpret_cast<const act_t*>(p.actions);
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t t_first = launch_t(p);

  // Warp tiles (32 lanes x V envs) are handed out by the global ticket counter, like the tiles of the step
  // kernel: faster warps take more, and the trip count stays warp-uniform so every lane reaches the votes.
  for (;;) {
    unsigned long long ticket = 0;
    if (lane == 0) ticket = atomicAdd(p.work_counter, 1ull) - p.work_base;
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    const uint64_t grp0 = ticket * 32;
    if (grp0 >= groups) break;
    const uint64_t grp = grp0 + lane;
    const bool active = FULL || grp < groups;
    const uint64_t base = p.first + (active ? grp * V : 0);
    Group<KIND, V> g;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      g.steps[v] = 0;
      g.sbt[v] = SBT_NONE;
      g.ret[v] = 0.0f;
#pragma unroll
      for (int c = 0; c < SD; ++c) g.st[v][c] = 0.0f;
    }
    if (active) {
#pragma unroll
      for (int c = 0; c < SD; ++c) {
        const Vec<float, V> s = ldv<float, V>(p.state + (uint64_t)c * p.ld + base);
#pragma unroll
        for (int v = 0; v < V; ++v) g.st[v][c] = s.v[v];
      }
      const Vec<cnt_t, V> cnt = ldv<cnt_t, V>(reinterpret_cast<const cnt_t*>(p.steps) + base);
#pragma unroll
      for (int v = 0; v < V; ++v) g.steps[v] = cnt_decode<CNT>(cnt.v[v], t_first);
      if constexpr (!AUTO && KIND == 0) {
        const Vec<uint32_t, V> sb = ldv<uint32_t, V>(p.sbt + base);
#pragma unroll
        for (int v = 0; v < V; ++v) g.sbt[v] = sb.v[v];
      }
      if (track_ret) {
        const Vec<float, V> er = ldv<float, V>(p.ep_return + base);
#pragma unroll
        for (int v = 0; v < V; ++v) g.ret[v] = er.v[v];
      }
    }
    if constexpr (PARAMS) {  // this thread's own slots: no synchronisation with other threads needed
#pragma unroll
      for (int c = 0; c < E::NP; ++c) {
        Vec<float, V> r;
#pragma unroll
        for (int v = 0; v < V; ++v) r.v[v] = 1.0f;  // inactive lanes step zero states with harmless constants
        if (active) r = ldv<float, V>(p.params + (uint64_t)c * p.ld + base);
#pragma unroll
        for (int v = 0; v < V; ++v) par_slots[c * V + v][threadIdx.x] = r.v[v];
      }
    }

    if constexpr (E::HAS_OBS_CACHE) {  // step_group<OBS_VALID> relies on g.obs from here on
#pragma unroll
      for (int v = 0; v < V; ++v) E::obs(g.st[v], g.obs[v]);
    }
    // Actions are staged ACT_RING steps ahead in shared memory with cp.async: every lane copies its own
    // 4 (uint8) or 16 (float) bytes of the row ACT_RING steps ahead and later reads back exactly those bytes, so no
    // cross-lane synchronisation is needed, only its own commit groups.  A load issued one step ahead into a
    // register (round 1, plus an L1 prefetch four rows ahead) arrived late under the write-heavy DRAM traffic of a
    // rollout: 10-25 % of all stall samples sat on the first use of the action word (profiles/README.md).
    constexpr bool STAGED = V == 4;  // scalar lanes (ragged sizes) load the row at its use
    [[maybe_unused]] uint32_t ring_addr = 0;
    const act_t* act_ptr = actions ? actions + base : nullptr;  // row being fetched next
    if constexpr (STAGED) {
      ring_addr = tma::smem_u32(&act_ring[0][threadIdx.x * V]);
      if (!policy) {
#pragma unroll
        for (int j = 0; j < ACT_RING; ++j) {
          if (active && (uint32_t)j < p.K) {
            cp_async<sizeof(act_t) * V>(ring_addr + j * RING_STRIDE, act_ptr);
            act_ptr += p.ld;
          }
          cp_async_commit();  // one group per row, empty or not: the wait below counts groups
        }
      }
    }

    // Sum of the lengths of the episodes an env finishes during this launch = steps_before + K - steps_after,
    // so the per-step tally is not needed here (counters saturate only after 4e9 steps).
    uint32_t steps_before = 0;
    if constexpr (AUTO) {
#pragma unroll
      for (int v = 0; v < V; ++v) steps_before += g.steps[v];
    }

    // running output pointers: one 64-bit add per array per step instead of a multiply-add chain per store
    const uint64_t obs_step = (uint64_t)OD * p.ld;
    float* obs_ptr = (FULL || p.obs_out) ? p.obs_out + base : nullptr;
    float* rew_ptr = (FULL || p.reward_out) ? p.reward_out + base : nullptr;
    uint8_t* flg_ptr = (FULL || p.flags_out) ? p.flags_out + base : nullptr;

    // One step of this warp tile.  `trusted_tag` selects the form without per-step precondition tests; the
    // return value says whether the invariant behind it still holds (it can only break when a reset state
    // comes from an injected pool, and is re-checked right there, under the same rare branch).
    ResetPrefetch pre;
    [[maybe_unused]] uint32_t redrawn = 0;  // REDRAW: slots whose parameters were redrawn in this tile
    // Redraws slot `slot` of EVERY lane (full warp): the state the lane's env in that slot restarts from when its
    // current episode ends.  t_next = index of the next step to run; g.steps = counts at its entry.
    [[maybe_unused]] auto draw_ahead = [&](uint32_t slot, uint64_t t_next) {
      uint32_t count = g.steps[0];
#pragma unroll
      for (int v = 1; v < V; ++v) count = ((uint32_t)v == slot) ? g.steps[v] : count;
      float ns[4] = {0.0f, 0.0f, 0.0f, 0.0f}, full[SD];
      E::reset(philox_env(p.keys, p.env_base + base + slot, t_next - (uint64_t)count, TAG_AUTO_RESET), full);
#pragma unroll
      for (int c = 0; c < SD && c < 4; ++c) ns[c] = full[c];
      pre.smem[slot * 256] = make_float4(ns[0], ns[1], ns[2], ns[3]);
      pre.valid |= 1u << slot;
    };
    if constexpr (PREFETCH) {
      static_assert(SD <= 4, "one float4 per env");
      pre.smem = &next_reset[0][threadIdx.x];
    }
    // the actions of step `row`: out of the ring (and the row ACT_RING steps later starts on its way into the slot
    // just read), or straight from global memory for scalar lanes
    auto fetch_row = [&](RawActions<act_t, V>& dst, uint32_t row) {
      dst.zero();
      if (policy) return;
      if constexpr (STAGED) {
        cp_async_wait<ACT_RING - 1>();  // all but the ACT_RING - 1 newest groups have landed: row `row` is here
        const uint32_t slot = ring_addr + (row & (ACT_RING - 1)) * RING_STRIDE;
        if (active) dst.load_shared(slot);
        if (active && row + ACT_RING < p.K) {
          cp_async<sizeof(act_t) * V>(slot, act_ptr);
          act_ptr += p.ld;
        }
        cp_async_commit();
      } else {
        if (active) dst.load(act_ptr);
        act_ptr += p.ld;
      }
    };
    auto one_step = [&](auto trusted_tag, uint32_t kk, const RawActions<act_t, V>& a_cur) -> bool {
      constexpr bool TRUSTED = decltype(trusted_tag)::value;
      bool still = true;
      const uint64_t t = t_first + kk;
      act_t action[V];
      if (policy) {
        // Space::sample: one Philox block serves 4 consecutive envs (global group g >> 2)
        if constexpr (V == 4) {
          const uint4 w = philox_env(p.keys, (p.env_base + base) >> 2, t, TAG_ACTION);
          action[0] = action_from_word<KIND>(w.x);
          action[1] = action_from_word<KIND>(w.y);
          action[2] = action_from_word<KIND>(w.z);
          action[3] = action_from_word<KIND>(w.w);
        } else {
          const uint64_t gid = p.env_base + base;
          const uint4 w = philox_env(p.keys, gid >> 2, t, TAG_ACTION);
          const uint32_t lane_word = (gid & 2) ? ((gid & 1) ? w.w : w.z) : ((gid & 1) ? w.y : w.x);
          action[0] = action_from_word<KIND>(lane_word);
        }
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) action[v] = a_cur.get(v);
      }
      PR prm;
      if constexpr (PARAMS) {
        // volatile loads: re-read every step, not hoisted into registers for the whole loop
#pragma unroll
        for (int c = 0; c < E::NP; ++c) {
#pragma unroll
          for (int v = 0; v < V; ++v) prm.r[c][v] = *static_cast<volatile const float*>(&par_slots[c * V + v][threadIdx.x]);
        }
      }
      step_group<KIND, V, AUTO, false, false, RESET_BY_CALLER, TRUSTED, true, PR>(p, active, base, t, action, track_ret,
                                                                                  g, acc, prm);

      // ---- trajectory stores (before the resets: reward and flags belong to the finishing step; the
      // observation is stored after them, it is the post-reset one) ----
      const uint32_t w = packed_flags<KIND, V>(g);
      if (active) {
        if (FULL || rew_ptr) {
          Vec<float, V> rw;
#pragma unroll
          for (int v = 0; v < V; ++v) rw.v[v] = g.reward[v];
          stv<float, V>(rew_ptr, rw);
          rew_ptr += p.ld;
        }
        if (FULL || flg_ptr) {
          if constexpr (V == 4) {
            *reinterpret_cast<uint32_t*>(flg_ptr) = w;
          } else {
            *flg_ptr = (uint8_t)w;
          }
          flg_ptr += p.ld;
        }
      }

      // ---- finished envs: one warp vote, then statistics + resets only where needed ----
      const uint32_t wf = active ? w : 0u;
      if (__ballot_sync(0xffffffffu, wf != 0u) != 0u) {
        dones += __popc((wf | (wf >> 1)) & 0x01010101u);
        if constexpr (AUTO) {
          tally_packed<KIND, V, false>(wf, g, acc);
          uint32_t pending = 0;
#pragma unroll
          for (int v = 0; v < V; ++v) pending |= ((wf >> (8 * v)) & 0xffu) ? (1u << v) : 0u;
          if constexpr (FINAL) {  // g.st / g.obs still hold what the finishing step produced
#pragma unroll
            for (int v = 0; v < V; ++v) {
              if (pending & (1u << v)) {
                float* dst = p.final_obs_out + (uint64_t)kk * OD * p.ld + base + v;
#pragma unroll
                for (int c = 0; c < OD; ++c) dst[(uint64_t)c * p.ld] = E::OBS_IS_STATE ? g.st[v][c < SD ? c : 0] : g.obs[v][c];
              }
            }
          }
          if constexpr (PREFETCH) {
            // Slots about to be consumed whose state is not there (never drawn in this tile, or consumed since):
            // redraw those slots for the WHOLE warp, so that the divergent pass below only ever picks states up.
            // In steady state a slot is redrawn every ~10 steps (an env must finish twice in between).
            if (!p.reset_pool) {
              uint32_t need = __reduce_or_sync(0xffffffffu, pending & ~pre.valid);
              while (need) {
                const uint32_t slot = __ffs(need) - 1;
                need &= need - 1;
                draw_ahead(slot, t + 1);
              }
            }
          }
          if constexpr (REDRAW) {  // into this thread's slots: the next step of the tile reads them
            redrawn |= pending;
            redraw_pending<KIND, V>(p, base, t, pending, g, RedrawDst{&par_slots[0][threadIdx.x], (uint64_t)V * 256, 256});
          }
          reset_pending<KIND, V>(p, base, t, pending, g, PREFETCH ? &pre : nullptr);
          if constexpr (TRUSTED && E::HAS_TRUSTED) {
            if (p.reset_pool) still = __all_sync(0xffffffffu, group_trusted<KIND, V>(g));
          }
        }
      }

      if (active && (FULL || obs_ptr)) {
#pragma unroll
        for (int c = 0; c < OD; ++c) {
          Vec<float, V> o;
#pragma unroll
          for (int v = 0; v < V; ++v) o.v[v] = E::OBS_IS_STATE ? g.st[v][c < SD ? c : 0] : g.obs[v][c];
          stv<float, V>(obs_ptr + (uint64_t)c * p.ld, o);
        }
        obs_ptr += obs_step;
      }
      return still;
    };
    bool trusted = false;  // warp-uniform
    if constexpr (E::HAS_TRUSTED) trusted = __all_sync(0xffffffffu, group_trusted<KIND, V>(g));  // zeros (inactive) pass
    auto step_any = [&](uint32_t kk, const RawActions<act_t, V>& a_cur) {
      if constexpr (E::HAS_TRUSTED) {
        if (trusted) {
          if constexpr (E::CONTINUOUS) {
            // a NaN action would break the invariant: the sum of the lane's actions is NaN iff one of them is
            // (or +inf meets -inf, which only costs this one checked step); such a step runs checked, and the
            // invariant is tested again after it
            if (!policy) {
              float sum = a_cur.get(0);
#pragma unroll
              for (int v = 1; v < V; ++v) sum += a_cur.get(v);
              if (__any_sync(0xffffffffu, sum != sum)) {
                one_step(std::false_type{}, kk, a_cur);
                trusted = __all_sync(0xffffffffu, group_trusted<KIND, V>(g));
                return;
              }
            }
          }
          trusted = one_step(std::true_type{}, kk, a_cur);
          return;
        }
      }
      one_step(std::false_type{}, kk, a_cur);
    };
#pragma unroll 1
    for (uint32_t kk = 0; kk < p.K; ++kk) {
      RawActions<act_t, V> a_cur;
      fetch_row(a_cur, kk);
      step_any(kk, a_cur);
    }
    if constexpr (STAGED) {
      if (!policy) cp_async_wait<0>();  // the ring is reused by this warp's next tile
    }
    if constexpr (AUTO) {
      if (active) {
        uint32_t steps_after = 0;
#pragma unroll
        for (int v = 0; v < V; ++v) steps_after += g.steps[v];
        acc.length_sum += (unsigned long long)steps_before + (unsigned long long)V * p.K - steps_after;
      }
    }

    if (active) {
#pragma unroll
      for (int c = 0; c < SD; ++c) {
        Vec<float, V> s;
#pragma unroll
        for (int v = 0; v < V; ++v) s.v[v] = g.st[v][c];
        stv<float, V>(p.state + (uint64_t)c * p.ld + base, s);
      }
      Vec<cnt_t, V> cnt;
#pragma unroll
      for (int v = 0; v < V; ++v) cnt.v[v] = cnt_encode<CNT>(g.steps[v], t_first + p.K);
      stv<cnt_t, V>(reinterpret_cast<cnt_t*>(p.steps) + base, cnt);
      if constexpr (!AUTO && KIND == 0) {
        Vec<uint32_t, V> sb;
#pragma unroll
        for (int v = 0; v < V; ++v) sb.v[v] = g.sbt[v];
        stv<uint32_t, V>(p.sbt + base, sb);
      }
      if (track_ret) {
        Vec<float, V> er;
#pragma unroll
        for (int v = 0; v < V; ++v) er.v[v] = g.ret[v];
        stv<float, V>(p.ep_return + base, er);
      }
      if constexpr (REDRAW) {  // the parameters of the episodes that run on past this launch, if any were drawn
        if (redrawn) {
#pragma unroll
          for (int c = 0; c < E::NP; ++c) {
            Vec<float, V> r;
#pragma unroll
            for (int v = 0; v < V; ++v) r.v[v] = par_slots[c * V + v][threadIdx.x];
            stv<float, V>(const_cast<float*>(p.params) + (uint64_t)c * p.ld + base, r);
          }
        }
      }
    }
  }
  acc.done_steps = dones;
  stats_flush<KIND>(acc, p);
  fused_clock_advance(p);
}

// =============================================================================================
// cold kernels: reset, observation, action sampling, counter conversion
// =============================================================================================
// Gym::reset of env i (cartpole.rs:238-249, mountain_car.rs:279-291): new state, counters cleared, observation out
template <int KIND, int CNT>
__device__ __forceinline__ void reset_one(const KernelParams& p, uint64_t i, uint64_t reset_index) {
  using E = Env<KIND>;
  using cnt_t = typename CounterType<CNT>::type;
  float st[E::SD], obs[E::OD];
  const uint64_t g = p.env_base + i;
  if (p.reset_pool) {
    const uint64_t j = (g + reset_index) % p.pool_len;
#pragma unroll
    for (int c = 0; c < E::SD; ++c) st[c] = p.reset_pool[(uint64_t)c * p.pool_len + j];
  } else {
    E::reset(philox_env(p.seed, g, reset_index, TAG_RESET), st);
  }
#pragma unroll
  for (int c = 0; c < E::SD; ++c) p.state[(uint64_t)c * p.ld + i] = st[c];
  reinterpret_cast<cnt_t*>(p.steps)[i] = cnt_encode<CNT>(0u, launch_t(p));  // cartpole.rs:243
  if (p.sbt) p.sbt[i] = SBT_NONE;                                            // cartpole.rs:239
  if (p.ep_return) p.ep_return[i] = 0.0f;
  if (p.obs_out) {
    E::obs(st, obs);
#pragma unroll
    for (int c = 0; c < E::OD; ++c) p.obs_out[(uint64_t)c * p.ld + i] = obs[c];
  }
}

template <int KIND, int CNT>
__global__ void reset_kernel(const KernelParams p, const uint8_t* mask, uint64_t reset_index) {
  using E = Env<KIND>;
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.n) return;
  const uint64_t i = p.first + j;
  if (mask && !mask[i]) {
    if (p.obs_out) {
      float st[E::SD], obs[E::OD];
#pragma unroll
      for (int c = 0; c < E::SD; ++c) st[c] = p.state[(uint64_t)c * p.ld + i];
      E::obs(st, obs);
#pragma unroll
      for (int c = 0; c < E::OD; ++c) p.obs_out[(uint64_t)c * p.ld + i] = obs[c];
    }
    return;
  }
  reset_one<KIND, CNT>(p, i, reset_index);
}

// Masked reset without an observation output -- the caller's `if done { env.reset() }` after a manual-mode step
// (cartpole.rs:468-470), where few envs are selected: each thread scans 16 mask bytes with one 128-bit load and
// only then touches the envs whose byte is set (the one-thread-per-env form spends its time on 1-byte loads).
// Requires first == 0, n % 16 == 0 and a 16-byte-aligned mask.
template <int KIND, int CNT>
__global__ void __launch_bounds__(256) reset_sparse_kernel(const KernelParams p, const uint8_t* mask, uint64_t reset_index) {
  // Each warp scans 512 envs (one 128-bit mask load per lane), queues the selected ones in shared memory and
  // then resets them with all lanes busy, whatever their distribution over the lanes' 16-env spans.
  __shared__ uint16_t queue[8][512];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // 16-env span of this lane
  uint4 m = make_uint4(0u, 0u, 0u, 0u);
  if (j * 16 < p.n) m = reinterpret_cast<const uint4*>(mask)[j];
  const uint32_t words[4] = {m.x, m.y, m.z, m.w};
  uint32_t bits = 0;  // bit b = env b of the span is selected
#pragma unroll
  for (int b = 0; b < 16; ++b) bits |= ((words[b >> 2] >> (8 * (b & 3))) & 0xffu) ? (1u << b) : 0u;
  if (__ballot_sync(0xffffffffu, bits != 0u) == 0u) return;
  // exclusive prefix sum of the per-lane counts
  const uint32_t mine = __popc(bits);
  uint32_t incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= (uint32_t)o) incl += up;
  }
  const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
  uint32_t pos = incl - mine;
  for (uint32_t rest = bits; rest; rest &= rest - 1) queue[warp][pos++] = (uint16_t)(lane * 16 + (__ffs(rest) - 1));
  __syncwarp();
  const uint64_t warp_base = (j - lane) * 16;
  for (uint32_t k = lane; k < total; k += 32) reset_one<KIND, CNT>(p, warp_base + queue[warp][k], reset_index);
}

template <int KIND>
__global__ void obs_kernel(const float* state, float* obs_out, uint64_t n) {
  using E = Env<KIND>;
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float st[E::SD], obs[E::OD];
#pragma unroll
  for (int c = 0; c < E::SD; ++c) st[c] = state[(uint64_t)c * n + i];
  E::obs(st, obs);
#pragma unroll
  for (int c = 0; c < E::OD; ++c) obs_out[(uint64_t)c * n + i] = obs[c];
}

// device clock: t += dt, ticket base += tickets (one thread, enqueued after the launches of a call)
__global__ void clock_advance_kernel(unsigned long long* clock, unsigned long long dt, unsigned long long tickets) {
  clock[0] += dt;
  clock[1] += tickets;
}

template <int KIND>
__global__ void sample_actions_kernel(typename Env<KIND>::act_t* out, uint64_t n, uint64_t seed, uint64_t env_base,
                                      uint64_t t, const unsigned long long* t_dev) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (t_dev) t = *t_dev;
  const uint64_t g = env_base + i;
  const uint4 w = philox_env(seed, g >> 2, t, TAG_ACTION);
  const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
  out[i] = action_from_word<KIND>(ws[g & 3]);
}

// episode step counts (uint32, what mgym_set_state / mgym_get_state exchange) <-> the handle's own representation
template <int CNT>
__global__ void counters_from_steps_kernel(const uint32_t* steps_or_null, typename CounterType<CNT>::type* out, uint64_t n,
                                           uint64_t t, const unsigned long long* t_dev) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t_dev) t = *t_dev;
  if (i < n) {
    uint32_t steps = steps_or_null ? steps_or_null[i] : 0u;
    // a 16-bit representation exists only below a time limit <= 65535: an injected count beyond it means "past the
    // limit" whatever its value, and must not wrap around to "young episode"
    if constexpr (sizeof(typename CounterType<CNT>::type) == 2) steps = min(steps, 0xFFFFu);
    out[i] = cnt_encode<CNT>(steps, t);
  }
}
template <int CNT>
__global__ void steps_from_counters_kernel(const typename CounterType<CNT>::type* in, uint32_t* steps, uint64_t n,
                                           uint64_t t, const unsigned long long* t_dev) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t_dev) t = *t_dev;
  if (i < n) steps[i] = cnt_decode<CNT>(in[i], t);
}

// ---- per-env parameters (mgym_set_params / mgym_sample_params / mgym_get_params) ----------------------------------
struct ParamVec {
  float v[MAX_PARAMS];
};

// Is every parameter finite, and every parameter c with bit c of `positive` set > 0?  Runs before anything is
// copied into the handle, like validate_actions_kernel.
__global__ void validate_params_kernel(const float* params, uint64_t n, int np, uint32_t positive, uint32_t* bad) {
  bool mine = false;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (uint64_t)np * n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    const float x = params[i];
    const uint32_t c = (uint32_t)(i / n);
    mine |= !isfinite(x) || (((positive >> c) & 1u) && !(x > 0.0f));
  }
  if (__any_sync(0xffffffffu, mine) && (threadIdx.x & 31) == 0) *bad = 1u;
}

__global__ void fill_params_kernel(float* out, uint64_t n, int np, ParamVec value) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int c = 0; c < np; ++c) out[(uint64_t)c * n + i] = value.v[c];
}

// Parameter c of env i (global index g = env_base + i) is word c % 4 of the Philox block with counter (g, key) and
// tag TAG_PARAMS + c / 4, mapped to U[lo, lo + range) as the reset states are: independent of sharding and launch
// geometry.  mask (device [n] or null): only envs with mask[i] != 0 are redrawn.
__global__ void sample_params_kernel(float* params, uint64_t n, int np, const uint8_t* mask, uint64_t seed,
                                     uint64_t env_base, uint64_t key, ParamBox box) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (mask && !mask[i])) return;
  const uint64_t g = env_base + i;
  for (int b = 0; b * 4 < np; ++b) {
    const uint4 w = philox_env(seed, g, key, TAG_PARAMS + (uint32_t)b);
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 4 * b + j;
      if (c < np) params[(uint64_t)c * n + i] = uniform_f64_to_f32(ws[j], box.lo[c], box.range[c]);
    }
  }
}

// Explicit resets of a handle with redraw ranges (mgym_reset / mgym_reset_masked), after the reset kernel: the
// parameters of every reset env (mask[i] != 0, or all with mask == null) from the Philox blocks with the counter of
// its reset state, (g, reset call index), and tags TAG_REDRAW_RESET + c / 4.  Cold: one thread per env.
__global__ void reset_redraw_params_kernel(float* params, uint64_t n, int np, const uint8_t* mask, uint64_t seed,
                                           uint64_t env_base, uint64_t reset_index, ParamBox box) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (mask && !mask[i])) return;
  const uint64_t g = env_base + i;
  for (int b = 0; b * 4 < np; ++b) {
    const uint4 w = philox_env(seed, g, reset_index, TAG_REDRAW_RESET + (uint32_t)b);
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 4 * b + j;
      if (c < np) params[(uint64_t)c * n + i] = uniform_f64_to_f32(ws[j], box.lo[c], box.range[c]);
    }
  }
}

// validate_actions: is every discrete action inside Discrete(num_actions)?  Runs BEFORE the step, so an invalid
// batch leaves the handle untouched (the reference asserts before any mutation, cartpole.rs:252)
__global__ void validate_actions_kernel(const uint8_t* actions, uint64_t count, uint32_t num_actions, uint32_t* bad) {
  bool mine = false;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x)
    mine |= actions[i] >= num_actions;
  if (__any_sync(0xffffffffu, mine) && (threadIdx.x & 31) == 0) *bad = 1u;
}

__global__ void fill_u32_kernel(uint32_t* out, uint32_t value, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = value;
}

// stats counters -> 5 doubles (the vector a host layer all-reduces)
__global__ void stats_export_kernel(const unsigned long long* stats, double* out) {
  if (threadIdx.x < 4) out[threadIdx.x] = (double)stats[threadIdx.x];
  if (threadIdx.x == 4) out[4] = *reinterpret_cast<const double*>(&stats[4]);
}

// exposes sin_ref / cos_ref for the parity tests (tests/test_gpu_trig.py)
__global__ void trig_probe_kernel(const float* x, float* s, float* c, float* s_only, float* c_only, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float sv, cv;
  sincos_ref(x[i], sv, cv);
  s[i] = sv;
  c[i] = cv;
  s_only[i] = sin_ref(x[i]);
  c_only[i] = cos_ref(x[i]);
}

// fast forms vs reference forms, counted on the device (tests/test_gpu_fastpath.py)
//   mode 0: fdiv_const_fast(x, c, rc) vs __fdiv_rn(x, c) for every bit pattern x in [first, first+n) with div_safe(x)
//   mode 1: sincos_small vs sincos_ref for every bit pattern with abstop12 < 0x3f4
//   mode 2: cos_fast vs cos_ref for every bit pattern with abstop12 < 0x42f
//   mode 3: fmod_fast(x, 2 pi) vs fmodf for every |x| < 2^22;  mode 4: sincos_fast vs sincos_ref, |x| < 120
__global__ void fast_exhaustive_kernel(int mode, uint64_t first, uint64_t n, float c, float rc,
                                       unsigned long long* checked, unsigned long long* bad, uint32_t* first_bad) {
  unsigned long long my_checked = 0, my_bad = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t u = (uint32_t)(first + i);
    const float x = __uint_as_float(u);
    bool mismatch = false, applicable = false;
    if (mode == 0) {
      applicable = div_safe(x);
      if (applicable) mismatch = __float_as_uint(fdiv_const_fast(x, c, rc)) != __float_as_uint(__fdiv_rn(x, c));
    } else if (mode == 1) {
      applicable = abstop12(x) < 0x3f4;
      if (applicable) {
        float s0, c0, s1, c1;
        sincos_small(x, s0, c0);
        sincos_ref(x, s1, c1);
        mismatch = __float_as_uint(s0) != __float_as_uint(s1) || __float_as_uint(c0) != __float_as_uint(c1);
      }
    } else if (mode == 2) {
      applicable = abstop12(x) < 0x42f;
      if (applicable) mismatch = __float_as_uint(cos_fast(x)) != __float_as_uint(cos_ref(x));
    } else if (mode == 3) {  // fmod_fast(t, 2 pi) vs fmodf, |t| < 2^22
      applicable = fabsf(x) < 4194304.0f;
      if (applicable)
        mismatch = __float_as_uint(fmod_fast(x, TWO_PI_F, 0.15915494309189535f)) != __float_as_uint(fmodf(x, TWO_PI_F));
    } else {  // sincos_fast vs sincos_ref, |x| < 120
      applicable = abstop12(x) < 0x42f;
      if (applicable) {
        float s0, c0, s1, c1;
        sincos_fast(x, s0, c0);
        sincos_ref(x, s1, c1);
        mismatch = __float_as_uint(s0) != __float_as_uint(s1) || __float_as_uint(c0) != __float_as_uint(c1);
      }
    }
    my_checked += applicable ? 1 : 0;
    if (mismatch) {
      my_bad += 1;
      atomicMin(first_bad, u);
    }
  }
  atomicAdd(checked, my_checked);
  if (my_bad) atomicAdd(bad, my_bad);
}

// fdiv_fast(a, b) vs __fdiv_rn(a, b) on pairs drawn from Philox, exponents spread over the safe range
__global__ void fast_div_random_kernel(uint64_t seed, uint64_t n, unsigned long long* checked, unsigned long long* bad) {
  unsigned long long my_checked = 0, my_bad = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint4 w = philox_env(seed, i, 0, 7u);
    const uint32_t pats[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float a = __uint_as_float(pats[2 * j]), b = __uint_as_float(pats[2 * j + 1]);
      // also the CartPole-shaped pair: any numerator over a denominator in [0.62, 0.67]
      const float b2 = 0.62f + 0.05f * ((pats[2 * j + 1] >> 8) * 0x1p-24f);
      if (div_safe(a) && div_safe(b)) {
        my_checked++;
        my_bad += __float_as_uint(fdiv_fast(a, b)) != __float_as_uint(__fdiv_rn(a, b));
      }
      if (div_safe(a)) {
        my_checked++;
        my_bad += __float_as_uint(fdiv_fast(a, b2)) != __float_as_uint(__fdiv_rn(a, b2));
      }
    }
  }
  atomicAdd(checked, my_checked);
  if (my_bad) atomicAdd(bad, my_bad);
}

// CartPole's fast forms (scalar and packed pair) vs the reference form on random states drawn ACROSS the fast
// precondition (|theta| < 0.25, |theta_dot| < 10): whenever a fast form says ok its state must be the reference's
// bits, and inside the precondition it must say ok (the numerators are then provably div_safe, see Env<0>::fast_ok).
// out = {checked, bad, accepted}
__global__ void cartpole_fast_random_kernel(uint64_t seed, uint64_t n, EnvConsts k, unsigned long long* out) {
  unsigned long long my_checked = 0, my_bad = 0, my_ok = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    float st[2][4];
    uint8_t act[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const uint4 w = philox_env(seed, 2 * i + j, 0, 9u);
      // theta: uniform in (-0.3, 0.3), every 8th sample a raw bit pattern below 0.25 (tiny values, denormals);
      // theta_dot: uniform in (-12, 12); x, x_dot: wide
      const float u0 = (w.x >> 8) * 0x1p-24f, u1 = (w.y >> 8) * 0x1p-24f, u2 = (w.z >> 8) * 0x1p-24f, u3 = (w.w >> 8) * 0x1p-24f;
      st[j][0] = (u0 - 0.5f) * 6.0f;
      st[j][1] = (u1 - 0.5f) * 20.0f;
      st[j][2] = ((w.x & 7u) == 0u) ? __uint_as_float((w.z % 0x3e800000u) | (w.y << 31)) : (u2 - 0.5f) * 0.6f;
      st[j][3] = (u3 - 0.5f) * 24.0f;
      act[j] = (uint8_t)(w.w & 1u);
    }
    float ref[2][4], one[2][4], two[2][4], aux = 0.0f;
    bool ok1[2], ok2[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
#pragma unroll
      for (int c = 0; c < 4; ++c) ref[j][c] = one[j][c] = two[j][c] = st[j][c];
      Env<0>::dynamics(ref[j], act[j], k, aux);
      ok1[j] = Env<0>::dynamics_fast(one[j], act[j], k, aux);
    }
    Env<0>::dynamics_fast2(two[0], two[1], act[0], act[1], k, ok2[0], ok2[1]);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const bool inside = fabsf(st[j][2]) < 0.25f && fabsf(st[j][3]) < 10.0f;
      bool bad = inside != ok1[j] || inside != ok2[j];
      if (ok1[j] && ok2[j]) {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          bad |= __float_as_uint(one[j][c]) != __float_as_uint(ref[j][c]) || __float_as_uint(two[j][c]) != __float_as_uint(ref[j][c]);
      }
      my_checked += 1;
      my_bad += bad ? 1 : 0;
      my_ok += ok1[j] ? 1 : 0;
    }
  }
  atomicAdd(out, my_checked);
  if (my_bad) atomicAdd(out + 1, my_bad);
  atomicAdd(out + 2, my_ok);
}

// digest of (x, sin x, cos x) from sincos_ref over magnitudes first, first+stride, ... and both signs: the same
// order-independent sum as oracle_trig_checksum (tests/test_gpu_trig_exhaustive.py)
__device__ __forceinline__ unsigned long long trig_mix(uint32_t xb, uint32_t sb, uint32_t cb) {
  unsigned long long h = ((unsigned long long)sb << 32) | cb;
  h ^= (unsigned long long)xb * 0x9E3779B97F4A7C15ull;
  h *= 0xD6E8FEB86659FD93ull;
  h ^= h >> 32;
  return h;
}
__global__ void trig_checksum_kernel(uint32_t first, uint64_t count, uint32_t stride, unsigned long long* out) {
  unsigned long long sum = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t mag = first + (uint32_t)(i * stride);
#pragma unroll
    for (uint32_t sign = 0; sign < 2; ++sign) {
      const uint32_t xb = mag | (sign << 31);
      float s, c;
      sincos_ref(__uint_as_float(xb), s, c);
      sum += trig_mix(xb, __float_as_uint(s), __float_as_uint(c));
      // the single-result forms must agree with the pair
      if (__float_as_uint(sin_ref(__uint_as_float(xb))) != __float_as_uint(s) ||
          __float_as_uint(cos_ref(__uint_as_float(xb))) != __float_as_uint(c))
        sum += 1;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, sum);
}

__global__ void philox_probe_kernel(const uint32_t* ctr_key, uint32_t* out, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* ck = ctr_key + i * 6;
  const uint4 r = philox4x32_10(make_uint4(ck[0], ck[1], ck[2], ck[3]), ck[4], ck[5]);
  out[i * 4 + 0] = r.x, out[i * 4 + 1] = r.y, out[i * 4 + 2] = r.z, out[i * 4 + 3] = r.w;
}

}  // namespace mgym
