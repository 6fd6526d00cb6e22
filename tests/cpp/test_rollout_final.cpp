// Final observations of a fused rollout through the C++ host layer (include/mgym.hpp): GpuVecEnv::rollout_final
// against K calls of mgym_step with final_obs_out on a twin handle.  Built and run by tests/test_gpu_rollout_final.py;
// prints "ALL OK".
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

int main() {
  const uint64_t n = 4096;
  const uint32_t K = 64;
  const int od = 4;
  const uint32_t kSentinel = 0x7fa5a5a5u;
  auto a = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).seed(21).build();
  auto b = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).seed(21).build();
  a.reset();
  b.reset();

  std::mt19937 rng(5);
  std::vector<uint8_t> acts((size_t)K * n);
  for (auto& x : acts) x = (uint8_t)(rng() & 1u);
  uint8_t* d_acts = device<uint8_t>(acts.size());
  cudaMemcpy(d_acts, acts.data(), acts.size(), cudaMemcpyHostToDevice);

  // K per-call steps with dense final observations
  float* d_step_final = device<float>((size_t)K * od * n);
  uint8_t* d_step_flags = device<uint8_t>((size_t)K * n);
  bool steps_ok = true;
  for (uint32_t k = 0; k < K; ++k)
    steps_ok = steps_ok && mgym_step(a.handle(), d_acts + (size_t)k * n, nullptr, nullptr, d_step_flags + (size_t)k * n,
                                     d_step_final + (size_t)k * od * n, nullptr) == MGYM_OK;
  EXPECT(steps_ok, "K calls of mgym_step with final_obs_out");

  // one rollout_final over the same actions, into a sentinel-filled buffer
  float* d_obs = device<float>((size_t)K * od * n);
  float* d_rew = device<float>((size_t)K * n);
  uint8_t* d_flags = device<uint8_t>((size_t)K * n);
  float* d_final = device<float>((size_t)K * od * n);
  std::vector<uint32_t> fill((size_t)K * od * n, kSentinel);
  cudaMemcpy(d_final, fill.data(), sizeof(float) * fill.size(), cudaMemcpyHostToDevice);
  b.rollout_final(K, d_acts, d_obs, d_rew, d_flags, d_final);

  const auto sf = to_host(d_step_flags, (size_t)K * n), rf = to_host(d_flags, (size_t)K * n);
  EXPECT(sf == rf, "rollout_final flags equal the steps' flags");
  const auto step_final = to_host(d_step_final, (size_t)K * od * n);
  const auto got = to_host(d_final, (size_t)K * od * n);
  size_t finished = 0;
  bool match = true, untouched = true;
  for (uint32_t k = 0; k < K; ++k)
    for (uint64_t i = 0; i < n; ++i) {
      const bool done = rf[(size_t)k * n + i] != 0;
      finished += done ? 1 : 0;
      for (int c = 0; c < od; ++c) {
        const size_t j = ((size_t)k * od + c) * n + i;
        uint32_t g, w;
        std::memcpy(&g, &got[j], 4);
        std::memcpy(&w, &step_final[j], 4);
        if (done)
          match = match && g == w;
        else
          untouched = untouched && g == kSentinel;
      }
    }
  EXPECT(finished > n / 4 && match, "final observations of finished envs equal mgym_step's, bit for bit");
  EXPECT(untouched, "entries of live envs are not written");

  std::vector<float> sa, sb;
  std::vector<uint32_t> ca, cb, ba, bb;
  a.get_state(sa, ca, ba);
  b.get_state(sb, cb, bb);
  EXPECT(std::memcmp(sa.data(), sb.data(), sizeof(float) * sa.size()) == 0 && ca == cb, "the same state afterwards");

  bool threw = false;
  try {
    b.rollout_final(K, d_acts, d_obs, d_rew, d_flags, d_obs);
  } catch (const mgym::Error& e) {
    threw = e.code() == MGYM_ERR_BAD_ARGUMENT;
  }
  EXPECT(threw, "final_obs_traj == obs_traj throws");

  auto manual = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).auto_reset(false).build();
  manual.reset();
  threw = false;
  try {
    manual.rollout_final(K, d_acts, d_obs, d_rew, d_flags, d_final);
  } catch (const mgym::Error& e) {
    threw = e.code() == MGYM_ERR_BAD_ARGUMENT;
  }
  EXPECT(threw, "a manual-mode handle throws");

  cudaFree(d_acts), cudaFree(d_step_final), cudaFree(d_step_flags);
  cudaFree(d_obs), cudaFree(d_rew), cudaFree(d_flags), cudaFree(d_final);
  if (failures) {
    std::printf("%d FAILED\n", failures);
    return 1;
  }
  std::printf("ALL OK\n");
  return 0;
}
