/*
 * push_sampler.cpp — TEST HARNESS: the host build of sample_push (solorl_b200/csrc/solo_env.cuh), the random push
 * schedule of the env step, so that the `-m "not gpu"` suite can check the schedule and the GPU suite can compare
 * the device's pushes with it bit for bit.  Never built into the product.
 */
#include <string>

#include "../../include/solo_b200.h"
#include "../../solorl_b200/csrc/solo_core.cuh"
#include "../../solorl_b200/csrc/solo_env.cuh"
#include "../../solorl_b200/csrc/solo_host_model.h"

using namespace solo;

extern "C" {

/* out [n][T][3] = the push (fx, fy, 0) of control steps t0 .. t0+T-1 of episode `episode` of the envs with global
 * ids gid0 .. gid0+n-1.  Returns SOLO_E_ARG for push fields solo_create rejects. */
int push_sample(const SoloSimParams* p, uint64_t seed, int64_t gid0, int n, uint32_t episode, int32_t t0, int T,
                float* out) {
  PushParams pp;
  std::string err;
  const int rc = build_push_params(*p, pp, err);
  if (rc != 0) return rc;
  for (int i = 0; i < n; i++)
    for (int k = 0; k < T; k++) {
      const PushSample s = sample_push(pp, (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32), gid0 + i, episode,
                                       t0 + k);
      float* o = out + ((size_t)i * T + k) * 3;
      o[0] = s.fx; o[1] = s.fy; o[2] = 0.f;
    }
  return 0;
}

}  // extern "C"
