// Host-side launch of the step-based env kernel (fg_env_step.cu).
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "fancy_gym_b200.h"

namespace fg {

// Kernel-side copy of fg_env_step_cfg (passed by value as a __grid_constant__ kernel parameter).
struct EnvStepDev {
  double dt;        // python float 0.01
  float dt_f;       // float32(0.01): numpy's weak-scalar promotion when the action is float32
  int max_steps;    // <= 0: never truncates
  int allow_self, allow_wall, rew_fct;
  double penalty;
};

// Returns the CUDA error of the launch; *why is set (and nothing is launched) for a combination that is not instantiated.
cudaError_t launch_env_step(const EnvStepDev& c, int env_kind, int n_dof, bool a64, const fg_env_step_io& io, long long B,
                            cudaStream_t stream, const char** why);

}  // namespace fg
