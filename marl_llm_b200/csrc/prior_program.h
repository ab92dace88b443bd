// prior_program.h — what swarm_abi.cu needs of a loaded prior program (prior_abi.cu; DESIGN.md §12).
#pragma once
#include "../../include/swarm_b200.h"
#include "../../include/swarm_prior_api.cuh"

#include <cuda_runtime.h>

// entry points of a program's CUBIN (include/swarm_prior_api.cuh), in this order
enum { SWARM_PRIOR_F32, SWARM_PRIOR_F64, SWARM_PRIOR_ACTIONS, SWARM_PRIOR_ENTRIES };

int swarm_prior_program_device_(const swarm_prior_program *prog);
// launches entry `entry` of prog with `ctas` CTAs on the current device, k_prior's block size for n_a agents: CTA b serves env
// env_ids[b] (device), or env b when env_ids is NULL
int swarm_prior_program_launch_(const swarm_prior_program *prog, int entry, const swarm_prior_args &args, const int *env_ids,
                                int ctas, int n_a, cudaStream_t stream);

int swarm_prior_population_device_(const swarm_prior_population *pop);
int swarm_prior_population_envs_(const swarm_prior_population *pop);
// launches entry `entry` of every program of pop over its envs, in program order (none for a program without envs), adding the
// launches to *launches
int swarm_prior_population_launch_(const swarm_prior_population *pop, int entry, const swarm_prior_args &args, int n_a,
                                   cudaStream_t stream, int64_t *launches);
