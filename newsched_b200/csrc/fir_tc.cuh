// fir_tc.cuh -- internal interface of the tensor-core (tcgen05) block-Toeplitz FIR (fir_tc.cu), used by fir.cu
#pragma once
#include <cuda_runtime.h>

namespace b200 {
struct tc_plan;
// complex stream, real taps; decimation 1..8; up to 2048 taps per polyphase branch.  real = 1 (float stream):
// decimation 1 and up to 449 taps (the tap-stationary kernel, two 4096-sample runs per tile)
bool tc_supported(int n_taps, int decimation, int real);
int tc_create(const float* taps, int n_taps, int decimation, int real, int fuse, float kre, float kim, tc_plan** out);
void tc_destroy(tc_plan* p);
int tc_launch(tc_plan* p, const float* d_hist, const void* d_in, void* d_out, long long n_in,
              long long n_out, cudaStream_t s);
} // namespace b200
