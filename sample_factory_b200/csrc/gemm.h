// Internal interface between the GEMM engines of libsfb200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sfb {

constexpr int SFB_TC_UNSUPPORTED = -1000;   // shape/alignment not handled by the tcgen05 engine -> caller uses SIMT

// tcgen05 engine (gemm_tc.cu). Return 0, an error code, or SFB_TC_UNSUPPORTED.
int tc_linear_act_forward(const float* x, int64_t ldx, const float* W, const float* b, float* y, int64_t ldy, int64_t M,
                          int N, int K, int act, int engine, cudaStream_t st);
int tc_linear_heads_partials(int N, int A, int engine);
int tc_linear_act_heads_forward(const float* x, int64_t ldx, const float* W, const float* b, float* y, int64_t ldy,
                                int64_t M, int N, int K, int act, int engine, const float* Wv, const float* Wa, int A,
                                float* head_part, cudaStream_t st);
// colsum_part (optional, (M/32) * K floats): the dX GEMM's epilogue leaves per-warp column sums of dx there and sets
// *colsum_fused = 1 when it could (full tiles); the caller then only runs the fixed-order reduce over M/32 partial rows
int tc_linear_backward(const float* dz, int64_t lddz, const float* x, int64_t ldx, const float* W, int64_t M, int N,
                       int K, int act_prev, float* dW, float* dx, int64_t lddx, int engine, float* ws, cudaStream_t st,
                       float* colsum_part = nullptr, int* colsum_fused = nullptr);

}  // namespace sfb

namespace sfb {
// shared with the SIMT engine (gemm_simt.cu)
int choose_splits(int64_t M, int N, int K);
int splitk_reduce(const float* part, int splits, int64_t M, int N, float* C, int64_t ldc, cudaStream_t st);
int colsum_reduce(const float* part, int64_t groups, int N, float* out, cudaStream_t st);
}  // namespace sfb
