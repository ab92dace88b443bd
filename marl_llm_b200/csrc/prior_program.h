// prior_program.h — what swarm_abi.cu needs of a loaded prior program (prior_abi.cu; DESIGN.md §12).
#pragma once
#include "../../include/swarm_b200.h"
#include "../../include/swarm_prior_api.cuh"

#include <cuda_runtime.h>

// entry points of a program's CUBIN (include/swarm_prior_api.cuh), in this order
enum { SWARM_PRIOR_F32, SWARM_PRIOR_F64, SWARM_PRIOR_ACTIONS, SWARM_PRIOR_ENTRIES };

int swarm_prior_program_device_(const swarm_prior_program *prog);
// launches entry `entry` of prog over num_envs envs (one CTA each, k_prior's block size for n_a agents) on the current device
int swarm_prior_program_launch_(const swarm_prior_program *prog, int entry, const swarm_prior_args &args, int num_envs, int n_a,
                                cudaStream_t stream);
