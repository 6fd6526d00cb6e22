// The per-episode parameter redraw through the C++ host layer (include/mgym.hpp): set_param_redraw, param_redraw,
// clear_param_redraw, and the rows they drive.  Built and run by tests/test_gpu_param_redraw.py; prints "ALL OK".
#include <cmath>
#include <cstdio>
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

int main() {
  const uint64_t n = 4096;
  const int np = mgym::GpuVecEnv::num_params(MGYM_CARTPOLE_V1);
  std::vector<float> d(np);
  mgym_param_defaults(MGYM_CARTPOLE_V1, d.data());
  std::vector<float> lo(np), hi(np);
  for (int c = 0; c < np; ++c) lo[c] = 0.8f * d[c], hi[c] = 1.2f * d[c];

  auto env = mgym::GpuVecEnv::builder(MGYM_CARTPOLE_V1, n).seed(11).build();
  env.reset();
  EXPECT(!env.param_redraw(), "no ranges on a new handle");
  env.set_param_redraw(lo, hi);
  std::vector<float> glo, ghi;
  EXPECT(env.param_redraw(&glo, &ghi) && glo == lo && ghi == hi, "param_redraw returns the ranges");
  std::vector<float> rows = env.get_params();
  bool defaults = true;
  for (int c = 0; c < np; ++c)
    for (uint64_t i = 0; i < n; ++i) defaults = defaults && rows[c * n + i] == d[c];
  EXPECT(defaults, "setting ranges leaves the current episodes on the defaults");

  env.reset();
  rows = env.get_params();
  bool inside = true, moved = false;
  for (int c = 0; c < np; ++c)
    for (uint64_t i = 0; i < n; ++i) {
      const float x = rows[c * n + i];
      inside = inside && x >= lo[c] && x <= hi[c];
      moved = moved || x != d[c];
    }
  EXPECT(inside && moved, "reset() draws every env's parameters inside the ranges");

  // rows change exactly where an episode ended
  std::vector<uint8_t> push(n, 1);
  bool only_finished = true;
  size_t finished = 0;
  for (int t = 0; t < 60; ++t) {
    const std::vector<float> before = env.get_params();
    const mgym::HostStepInfo info = env.step_host(push);
    const std::vector<float> after = env.get_params();
    for (uint64_t i = 0; i < n; ++i) {
      const bool done = info.done[i] || info.truncated[i];
      finished += done ? 1 : 0;
      for (int c = 0; c < np && !done; ++c) only_finished = only_finished && after[c * n + i] == before[c * n + i];
    }
  }
  EXPECT(only_finished && finished > n, "step_host redraws only the envs that finished");

  bool threw = false;
  std::vector<float> bad = hi;
  bad[2] = std::nanf("");
  try {
    env.set_param_redraw(lo, bad);
  } catch (const mgym::Error& e) {
    threw = e.code() == MGYM_ERR_BAD_ARGUMENT;
  }
  EXPECT(threw && env.param_redraw(&glo, &ghi) && ghi == hi, "a NaN bound throws and changes nothing");

  env.clear_param_redraw();
  EXPECT(!env.param_redraw(), "clear_param_redraw turns redraw off");
  const std::vector<float> kept = env.get_params();
  env.reset();
  EXPECT(env.get_params() == kept, "without ranges reset() leaves the rows alone");

  auto acro = mgym::GpuVecEnv::builder(MGYM_ACROBOT_V1, 128).build();
  threw = false;
  try {
    acro.set_param_redraw({}, {});
  } catch (const mgym::Error& e) {
    threw = true;
  }
  EXPECT(threw, "Acrobot has no parameters to redraw");

  if (failures) {
    std::printf("%d FAILED\n", failures);
    return 1;
  }
  std::printf("ALL OK\n");
  return 0;
}
