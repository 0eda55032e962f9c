// Host-side launch of the step-based env kernel (fg_env_step.cu).
#pragma once
#include <cuda_runtime.h>

#include "fancy_gym_b200.h"
#include "fg_device.cuh"

namespace fg {

// Returns the CUDA error of the launch; *why is set (and nothing is launched) for a combination that is not instantiated.
cudaError_t launch_env_step(const ReacherCfg& c, int env_kind, int n_dof, bool a64, const fg_env_step_io& io, long long B,
                            cudaStream_t stream, const char** why);

}  // namespace fg
