// Per-episode returns and lengths through the C++ host layer (include/mgym.hpp): GpuVecEnv::rollout_episodes against
// K calls of GpuVecEnv::step_episodes on a twin handle, and both against the statistics.  Built and run by
// tests/test_gpu_episodes.py; prints "ALL OK".
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "../../include/mgym.hpp"

static int failures = 0;
#define EXPECT(cond, what)                                     \
  do {                                                         \
    if (cond) {                                                \
      std::printf("ok %s\n", what);                            \
    } else {                                                   \
      std::printf("FAIL %s (%s:%d)\n", what, __FILE__, __LINE__); \
      ++failures;                                              \
    }                                                          \
  } while (0)

template <typename T>
static T* device(size_t count) {
  T* p = nullptr;
  if (cudaMalloc(reinterpret_cast<void**>(&p), sizeof(T) * count) != cudaSuccess) {
    std::printf("FAIL cudaMalloc\n");
    std::exit(1);
  }
  return p;
}

template <typename T>
static std::vector<T> to_host(const T* d, size_t count) {
  std::vector<T> h(count);
  cudaDeviceSynchronize();
  cudaMemcpy(h.data(), d, sizeof(T) * count, cudaMemcpyDeviceToHost);
  return h;
}

template <typename T>
static void fill(T* d, size_t count, uint32_t bits) {
  std::vector<uint32_t> h(count, bits);
  cudaMemcpy(d, h.data(), sizeof(T) * count, cudaMemcpyHostToDevice);
}

int main() {
  const uint64_t n = 4096;
  const uint32_t K = 64;
  const uint32_t kSentinel = 0x7fa5a5a5u;
  auto a = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).seed(22).build();
  auto b = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).seed(22).build();
  a.reset();
  b.reset();

  std::mt19937 rng(6);
  std::vector<uint8_t> acts((size_t)K * n);
  for (auto& x : acts) x = (uint8_t)(rng() & 1u);
  uint8_t* d_acts = device<uint8_t>(acts.size());
  cudaMemcpy(d_acts, acts.data(), acts.size(), cudaMemcpyHostToDevice);

  // K per-call steps, each into its own sentinel-filled row
  float* d_step_ret = device<float>((size_t)K * n);
  uint32_t* d_step_len = device<uint32_t>((size_t)K * n);
  fill(d_step_ret, (size_t)K * n, kSentinel);
  fill(d_step_len, (size_t)K * n, kSentinel);
  std::vector<uint8_t> step_flags((size_t)K * n);
  for (uint32_t k = 0; k < K; ++k) {
    auto info = a.step_episodes(d_acts + (size_t)k * n, d_step_ret + (size_t)k * n, d_step_len + (size_t)k * n);
    cudaMemcpy(step_flags.data() + (size_t)k * n, info.flags, n, cudaMemcpyDeviceToHost);
  }

  // one rollout_episodes over the same actions
  float* d_obs = device<float>((size_t)K * 4 * n);
  float* d_rew = device<float>((size_t)K * n);
  uint8_t* d_flags = device<uint8_t>((size_t)K * n);
  float* d_ret = device<float>((size_t)K * n);
  uint32_t* d_len = device<uint32_t>((size_t)K * n);
  fill(d_ret, (size_t)K * n, kSentinel);
  fill(d_len, (size_t)K * n, kSentinel);
  b.rollout_episodes(K, d_acts, d_obs, d_rew, d_flags, nullptr, d_ret, d_len);

  const auto rf = to_host(d_flags, (size_t)K * n);
  EXPECT(rf == step_flags, "rollout_episodes flags equal the steps' flags");
  const auto sr = to_host(d_step_ret, (size_t)K * n), rr = to_host(d_ret, (size_t)K * n);
  const auto sl = to_host(d_step_len, (size_t)K * n), rl = to_host(d_len, (size_t)K * n);
  EXPECT(std::memcmp(sr.data(), rr.data(), sizeof(float) * sr.size()) == 0 && sl == rl,
         "rollout_episodes outputs equal the steps', bit for bit");
  size_t finished = 0;
  unsigned long long length_sum = 0;
  bool untouched = true, cartpole_return = true;
  for (size_t j = 0; j < rf.size(); ++j) {
    uint32_t r;
    std::memcpy(&r, &rr[j], 4);
    if (rf[j]) {
      ++finished;
      length_sum += rl[j];
      cartpole_return = cartpole_return && rr[j] == (float)rl[j];
    } else {
      untouched = untouched && r == kSentinel && rl[j] == kSentinel;
    }
  }
  const mgym_stats_t s = b.stats();
  EXPECT(finished > n / 4 && finished == s.episodes && length_sum == s.length_sum && cartpole_return,
         "lengths and returns add up to the statistics");
  EXPECT(untouched, "entries of live envs are not written");

  auto manual = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).auto_reset(false).build();
  manual.reset();
  bool threw = false;
  try {
    manual.rollout_episodes(K, d_acts, d_obs, d_rew, d_flags, nullptr, d_ret, d_len);
  } catch (const mgym::Error& e) {
    threw = e.code() == MGYM_ERR_BAD_ARGUMENT;
  }
  EXPECT(threw, "a manual-mode handle throws");

  cudaFree(d_acts), cudaFree(d_step_ret), cudaFree(d_step_len);
  cudaFree(d_obs), cudaFree(d_rew), cudaFree(d_flags), cudaFree(d_ret), cudaFree(d_len);
  if (failures) {
    std::printf("%d FAILED\n", failures);
    return 1;
  }
  std::printf("ALL OK\n");
  return 0;
}
