// mgym.hpp -- C++17 host layer over the C ABI of mgym.h: the batched counterpart of the reference's
// `impl Gym for CartPoleV1 / MountainCarV0` (src/classic_control/cartpole.rs:234-357,
// mountain_car.rs:275-339 under /root/reference).  Header only; link libmgym.so and libcudart.
//
//   auto env = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, 1 << 24).seed(7).build();   // CartPoleV1::builder().build()
//   const float* obs = env.reset();                       // Gym::reset        -> device [obs_dim][N]
//   mgym::StepInfo info = env.step(actions_device);       // Gym::step         -> StepInfo{state, reward, flags}
//   auto space = env.observation_space();                 // Gym::observation_space
//
// Names and meanings follow the reference: builder options sutton_barto_reward / is_euler
// (cartpole.rs:39-40) and goal_velocity (mountain_car.rs:33); StepInfo{state, reward, done, truncated}
// (cartpole.rs:300-305), with done/truncated packed as bit0/bit1 of `flags`; Testable::set_state
// (cartpole.rs:444-446).  Errors are exceptions carrying the C status code; an invalid action, which the
// reference turns into a panic (cartpole.rs:252), is mgym::InvalidAction when validate_actions is on.
#pragma once

#include <cuda_runtime_api.h>

#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "mgym.h"

namespace mgym {

class Error : public std::runtime_error {
 public:
  Error(int code, const std::string& what) : std::runtime_error(what), code_(code) {}
  int code() const { return code_; }

 private:
  int code_;
};
class InvalidAction : public Error {
 public:
  using Error::Error;
};

inline void check(int rc) {
  if (rc == MGYM_OK) return;
  const std::string msg = "mgym error " + std::to_string(rc) + ": " + mgym_last_error();
  if (rc == MGYM_ERR_INVALID_ACTION) throw InvalidAction(rc, msg);
  throw Error(rc, msg);
}
inline void check_cuda(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw Error(MGYM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// modurl::spaces::{Discrete, BoxSpace} as the reference uses them (cartpole.rs:58-69)
struct Discrete {
  int n;
  bool contains(long long a) const { return a >= 0 && a < n; }
};
struct BoxSpace {
  std::vector<float> low, high;
  bool contains(const std::vector<float>& x) const {
    if (x.size() != low.size()) return false;
    for (size_t i = 0; i < x.size(); ++i)
      if (!(x[i] >= low[i] && x[i] <= high[i])) return false;
    return true;
  }
};

// StepInfo { state, reward, done, truncated } (cartpole.rs:300-305), batched, in device memory.
struct StepInfo {
  const float* state;    // [obs_dim][N]
  const float* reward;   // [N]
  const uint8_t* flags;  // [N]: bit0 = done (terminated), bit1 = truncated
};
// The same on the host (small N: tests, scalar adapters).
struct HostStepInfo {
  std::vector<float> state, reward;
  std::vector<uint8_t> done, truncated;
};

class GpuVecEnv {
 public:
  class Builder {
   public:
    Builder(int kind, uint64_t num_envs) : kind_(kind), n_(num_envs) { check(mgym_config_default(kind, &cfg_)); }
    Builder& device(int ordinal) { device_ = ordinal; return *this; }
    Builder& seed(uint64_t s) { seed_ = s; return *this; }
    Builder& sutton_barto_reward(bool v) { cfg_.sutton_barto_reward = v; return *this; }  // cartpole.rs:39
    Builder& is_euler(bool v) { cfg_.is_euler = v; return *this; }                        // cartpole.rs:40
    Builder& goal_velocity(float v) { cfg_.goal_velocity = v; return *this; }             // mountain_car.rs:33
    Builder& auto_reset(bool v) { cfg_.auto_reset = v; return *this; }
    Builder& max_episode_steps(int v) { cfg_.max_episode_steps = v; return *this; }
    Builder& validate_actions(bool v) { cfg_.validate_actions = v; return *this; }
    Builder& track_stats(bool v) { cfg_.track_stats = v; return *this; }
    // per-env running return, so that MountainCarContinuous / Pendulum statistics carry a return sum
    Builder& track_returns(bool v) { cfg_.track_returns = v; return *this; }
    Builder& env_index_base(uint64_t v) { cfg_.env_index_base = v; return *this; }
    // step index and tile tickets on the device: step / rollout / sample_actions become CUDA-graph-capturable
    Builder& graph_capturable(bool v) { cfg_.device_clock = v; return *this; }
    GpuVecEnv build() const { return GpuVecEnv(kind_, n_, device_, seed_, cfg_); }

   private:
    int kind_;
    uint64_t n_;
    int device_ = 0;
    uint64_t seed_ = 0;
    mgym_config cfg_{};
  };
  static Builder builder(int kind, uint64_t num_envs) { return Builder(kind, num_envs); }

  GpuVecEnv(GpuVecEnv&& o) noexcept { *this = std::move(o); }
  GpuVecEnv& operator=(GpuVecEnv&& o) noexcept {
    if (this != &o) {
      release();
      h_ = o.h_, kind_ = o.kind_, n_ = o.n_, device_ = o.device_, stream_ = o.stream_;
      obs_ = o.obs_, reward_ = o.reward_, flags_ = o.flags_, act_ = o.act_;
      o.h_ = nullptr, o.obs_ = nullptr, o.reward_ = nullptr, o.flags_ = nullptr, o.act_ = nullptr;
    }
    return *this;
  }
  GpuVecEnv(const GpuVecEnv&) = delete;
  GpuVecEnv& operator=(const GpuVecEnv&) = delete;
  ~GpuVecEnv() { release(); }

  uint64_t num_envs() const { return n_; }
  int obs_dim() const { return mgym_obs_dim(kind_); }
  int state_dim() const { return mgym_state_dim(kind_); }
  bool continuous() const { return mgym_action_is_continuous(kind_) != 0; }
  void set_stream(cudaStream_t s) { stream_ = s; }
  mgym_env* handle() { return h_; }

  // ---- Gym trait --------------------------------------------------------------------------------
  const float* reset() {  // cartpole.rs:238-249
    check(mgym_reset(h_, obs_, stream_));
    return obs_;
  }
  const float* reset(const uint8_t* mask_device) {
    check(mgym_reset_masked(h_, mask_device, obs_, stream_));
    return obs_;
  }
  // For kinds whose observation is the state (CartPole, MountainCar, MountainCarContinuous) StepInfo.state is
  // the resident state rows themselves: no separate observation buffer is written.
  bool obs_is_state() const { return mgym_obs_dim(kind_) == mgym_state_dim(kind_); }
  StepInfo step(const void* actions_device) {  // cartpole.rs:251-348
    const bool alias = obs_is_state();
    check(mgym_step(h_, actions_device, alias ? nullptr : obs_, reward_, flags_, nullptr, stream_));
    return StepInfo{alias ? mgym_state_ptr(h_) : obs_, reward_, flags_};
  }
  BoxSpace observation_space() const {  // cartpole.rs:350-352
    BoxSpace b{std::vector<float>(obs_dim()), std::vector<float>(obs_dim())};
    check(mgym_space_observation(kind_, b.low.data(), b.high.data()));
    return b;
  }
  Discrete action_space_discrete() const { return Discrete{mgym_num_actions(kind_)}; }  // cartpole.rs:354-356
  BoxSpace action_space_box() const {
    BoxSpace b{std::vector<float>(1), std::vector<float>(1)};
    check(mgym_space_action(kind_, b.low.data(), b.high.data()));
    return b;
  }

  // ---- the caller's step loop, fused (cartpole.rs:460-471) ----------------------------------------
  void rollout(uint32_t K, const void* actions_device, float* obs_traj, float* reward_traj, uint8_t* flags_traj,
               unsigned long long* done_count_device = nullptr) {
    check(mgym_rollout(h_, K, actions_device, obs_traj, reward_traj, flags_traj, done_count_device, stream_));
  }
  // rollout plus the observation each finished episode ended on: final_obs_traj [K][obs_dim][N] (device) is written
  // only where flags_traj != 0 (mgym_rollout_final); auto-reset handles only
  void rollout_final(uint32_t K, const void* actions_device, float* obs_traj, float* reward_traj, uint8_t* flags_traj,
                     float* final_obs_traj, unsigned long long* done_count_device = nullptr) {
    check(mgym_rollout_final(h_, K, actions_device, obs_traj, reward_traj, flags_traj, final_obs_traj,
                             done_count_device, stream_));
  }
  void sample_actions(void* actions_device) { check(mgym_sample_actions(h_, actions_device, stream_)); }

  // ---- Testable (cartpole.rs:436-447) and checkpointing ---------------------------------------------
  void set_state(const std::vector<float>& state_soa, const std::vector<uint32_t>* steps = nullptr,
                 const std::vector<uint32_t>* sbt = nullptr) {
    if (state_soa.size() != (size_t)state_dim() * n_) throw Error(MGYM_ERR_BAD_ARGUMENT, "set_state: wrong size");
    check(mgym_set_state(h_, state_soa.data(), steps ? steps->data() : nullptr, sbt ? sbt->data() : nullptr, stream_));
    sync();
  }
  void get_state(std::vector<float>& state_soa, std::vector<uint32_t>& steps, std::vector<uint32_t>& sbt) {
    state_soa.resize((size_t)state_dim() * n_), steps.resize(n_), sbt.resize(n_);
    check(mgym_get_state(h_, state_soa.data(), steps.data(), sbt.data(), stream_));
    sync();
  }
  // ---- per-env physics parameters (domain randomisation) ------------------------------------------------
  static int num_params(int kind) { return mgym_num_params(kind); }
  // params_soa: [P][N] on the host or the device; nullptr returns to the kind's constants
  void set_params(const float* params_soa) {
    check(mgym_set_params(h_, params_soa, stream_));
  }
  std::vector<float> get_params() {
    std::vector<float> v((size_t)mgym_num_params(kind_) * n_);
    check(mgym_get_params(h_, v.data(), stream_));
    return v;
  }
  // low, high: P values each; mask_device: uint8[N] or nullptr
  void sample_params(const std::vector<float>& low, const std::vector<float>& high,
                     const uint8_t* mask_device = nullptr, uint64_t key = 0) {
    if ((int)low.size() != mgym_num_params(kind_) || (int)high.size() != mgym_num_params(kind_))
      throw Error(MGYM_ERR_BAD_ARGUMENT, "sample_params: low and high need num_params values each");
    check(mgym_sample_params(h_, low.data(), high.data(), mask_device, key, stream_));
  }
  // per-episode redraw: every reset draws the env's parameters from [low, high) (num_params values each)
  void set_param_redraw(const std::vector<float>& low, const std::vector<float>& high) {
    if ((int)low.size() != mgym_num_params(kind_) || (int)high.size() != mgym_num_params(kind_))
      throw Error(MGYM_ERR_BAD_ARGUMENT, "set_param_redraw: low and high need num_params values each");
    check(mgym_set_param_redraw(h_, low.data(), high.data(), stream_));
  }
  void clear_param_redraw() { check(mgym_set_param_redraw(h_, nullptr, nullptr, stream_)); }
  // true and the ranges when the handle redraws; false (low, high untouched) otherwise
  bool param_redraw(std::vector<float>* low = nullptr, std::vector<float>* high = nullptr) const {
    const int np = mgym_num_params(kind_);
    std::vector<float> lo((size_t)(np > 0 ? np : 0)), hi(lo.size());
    int on = 0;
    check(mgym_get_param_redraw(h_, &on, lo.data(), hi.data()));
    if (on && low) *low = lo;
    if (on && high) *high = hi;
    return on != 0;
  }

  mgym_stats_t stats() {
    mgym_stats_t s{};
    check(mgym_stats_get(h_, &s, stream_));
    return s;
  }
  // Sum of the statistics over the ranks of `nccl_comm` (an ncclComm_t), left as 5 doubles {episodes, terminated,
  // truncated, length_sum, return_sum} in the caller's DEVICE buffer; the only collective of the path (SURVEY 8(e)).
  void stats_allreduce(void* nccl_comm, double* device_vec5) {
    check(mgym_stats_allreduce(h_, nccl_comm, device_vec5, stream_));
  }

  // ---- host-side conveniences ------------------------------------------------------------------------
  std::vector<float> reset_host() {
    reset();
    return download(obs_, (size_t)obs_dim() * n_);
  }
  template <typename Action>  // uint8_t for Discrete kinds, float for Box kinds
  HostStepInfo step_host(const std::vector<Action>& actions) {
    if (actions.size() != n_ || sizeof(Action) != (continuous() ? 4u : 1u))
      throw Error(MGYM_ERR_BAD_ARGUMENT, "step_host: actions must be uint8[N] (Discrete) or float[N] (Box)");
    HostStepInfo out;
    out.state.resize((size_t)obs_dim() * n_), out.reward.resize(n_);
    std::vector<uint8_t> flags(n_);
    check(mgym_step_host(h_, actions.data(), out.state.data(), out.reward.data(), flags.data(), stream_));
    out.done.resize(n_), out.truncated.resize(n_);
    for (size_t i = 0; i < n_; ++i) {
      out.done[i] = flags[i] & MGYM_FLAG_TERMINATED;
      out.truncated[i] = (flags[i] & MGYM_FLAG_TRUNCATED) >> 1;
    }
    return out;
  }
  void sync() { check_cuda(cudaStreamSynchronize(stream_), "cudaStreamSynchronize"); }

 private:
  GpuVecEnv(int kind, uint64_t n, int device, uint64_t seed, const mgym_config& cfg)
      : kind_(kind), n_(n), device_(device) {
    check(mgym_create(kind, n, device, seed, &cfg, &h_));
    check_cuda(cudaSetDevice(device), "cudaSetDevice");
    check_cuda(cudaMalloc(reinterpret_cast<void**>(&obs_), sizeof(float) * obs_dim() * n), "cudaMalloc obs");
    check_cuda(cudaMalloc(reinterpret_cast<void**>(&reward_), sizeof(float) * n), "cudaMalloc reward");
    check_cuda(cudaMalloc(reinterpret_cast<void**>(&flags_), n), "cudaMalloc flags");
  }
  std::vector<float> download(const float* dev, size_t count) {
    std::vector<float> v(count);
    check_cuda(cudaMemcpyAsync(v.data(), dev, sizeof(float) * count, cudaMemcpyDeviceToHost, stream_), "cudaMemcpyAsync");
    sync();
    return v;
  }
  void release() {
    if (h_) mgym_destroy(h_);
    if (obs_) cudaFree(obs_);
    if (reward_) cudaFree(reward_);
    if (flags_) cudaFree(flags_);
    if (act_) cudaFree(act_);
    h_ = nullptr, obs_ = nullptr, reward_ = nullptr, flags_ = nullptr, act_ = nullptr;
  }

  mgym_env* h_ = nullptr;
  int kind_ = 0;
  uint64_t n_ = 0;
  int device_ = 0;
  cudaStream_t stream_ = nullptr;
  float* obs_ = nullptr;
  float* reward_ = nullptr;
  uint8_t* flags_ = nullptr;
  void* act_ = nullptr;
};

}  // namespace mgym
