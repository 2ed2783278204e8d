// Batched acting: one environment step of the four nets (actor, target actor, critic, target critic) over B
// environments (r2d2_act_* in include/r2d2_b200.h).
#pragma once
#include "common.cuh"

namespace r2d2 {

struct Act;

int act_create(Act** out, int obs, int act, int hidden, int max_batch);
int act_destroy(Act* a);
int act_load(Act* a, const float* const params[4], cudaStream_t stream);
int act_step(Act* a, const float* obs, const float* state_in, float* state_out, float* mu, int B, cudaStream_t stream);
int act_status(Act* a, int* status, cudaStream_t stream);

}  // namespace r2d2
