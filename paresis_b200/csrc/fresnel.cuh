// The Fresnel propagator of csrc/fresnel.cu as other translation units of the library call it (the plan and kernel
// structures stay private to that file).
#pragma once
#include "common.cuh"

namespace paresis {

// paresis_fresnel_convolve without the argument checks, plus `sum` (nullable): *sum += the fp64 sum over the image of
// the |.|^2 values the call delivers (the ones it adds into `acc`).
int fresnel_convolve(paresis_fresnel_plan* p, const float2* wave_in, const paresis_fresnel_kernel* k, float2 phase,
                     float2* wave_out, float* acc, double* sum, cudaStream_t s);
// whether `k` was prepared for plans of p's size
bool fresnel_kernel_fits(const paresis_fresnel_plan* p, const paresis_fresnel_kernel* k);
void fresnel_plan_dims(const paresis_fresnel_plan* p, int* nx, int* ny);

}  // namespace paresis
