/*
 * dyn_sampler.cpp — TEST HARNESS: the host build of sample_env_dyn (solorl_b200/csrc/solo_env.cuh), the draw of
 * a randomised handle's per-env dynamics at a reset, so that the `-m "not gpu"` suite can check the sampler and
 * the GPU suite can compare the device's draws with it bit for bit.  Never built into the product.
 */
#include <string>

#include "../../include/solo_b200.h"
#include "../../solorl_b200/csrc/solo_core.cuh"
#include "../../solorl_b200/csrc/solo_env.cuh"
#include "../../solorl_b200/csrc/solo_host_model.h"

using namespace solo;

extern "C" {

/* out [n][3] = (friction, base mass scale, motor strength) drawn at the reset that starts episode `episode` of the
 * envs with global ids gid0 .. gid0+n-1.  Returns SOLO_E_ARG for ranges solo_create rejects. */
int dyn_sample(const SoloSimParams* p, uint64_t seed, int64_t gid0, int n, uint32_t episode, float* out) {
  EnvRanges r;
  std::string err;
  const int rc = build_env_ranges(*p, r, err);
  if (rc != 0) return rc;
  for (int i = 0; i < n; i++) {
    const EnvDyn d = sample_env_dyn(r, (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32), gid0 + i, episode);
    out[3 * i] = d.mu; out[3 * i + 1] = d.sm; out[3 * i + 2] = d.st;
  }
  return 0;
}

}  // extern "C"
