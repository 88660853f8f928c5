// Host launchers that one libicap source file calls in another (not part of the C ABI in include/icap.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// misc.cu
extern "C" int icap_copy2d(const void* src, int src_dtype, int64_t src_ld, void* dst, int dst_dtype, int64_t dst_ld,
                           int64_t rows, int64_t cols, int accumulate, void* stream);

// attention_mma.cu: tensor-core (mma.sync) attention for bf16 / head dim 64
bool icap_mha_mma_ok(int dtype, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv, int64_t ldq, int64_t ldk, int64_t ldv,
                     const void* q, const void* k, const void* v);
int icap_mha_fwd_mma(int64_t B, int64_t H, int64_t Lq, int64_t Lk, const void* q, int64_t ldq, const void* k,
                     int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo, const uint8_t* kvalid, int causal,
                     float p_drop, uint64_t seed, const int* seed_dev, cudaStream_t st, int kv_static = 0);
int icap_mha_bwd_mma(int64_t B, int64_t H, int64_t Lq, int64_t Lk, const void* q, int64_t ldq, const void* k,
                     int64_t ldk, const void* v, int64_t ldv, const void* dout, int64_t lddo, void* dq, int64_t lddq,
                     void* dk_out, int64_t lddk, void* dv_out, int64_t lddv, const uint8_t* kvalid, int causal,
                     float p_drop, uint64_t seed, const int* seed_dev, cudaStream_t st);

// gemm_simt.cu, gemm_tc.cu: the two halves of icap_gemm
int icap_gemm_f32_launch(int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                         const float* B, int64_t ldb, float* C, int64_t ldc, const float* bias, int epi,
                         const float* aux, int64_t ldaux, int accumulate, int split_k, cudaStream_t st);
int icap_gemm_bf16_launch(int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda,
                          const void* B, int64_t ldb, void* C, int64_t ldc, int c_dtype, const float* bias, int epi,
                          const void* aux, int64_t ldaux, int accumulate, int split_k, cudaStream_t st);

// gemm_small.cu: the small-footprint bf16 GEMM for latency-bound shapes
unsigned long long* icap_trace_slot();
bool icap_gemm_small_eligible(int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, int c_dtype, int epi,
                              int accumulate, int split_k, const void* C, int64_t ldc);
int icap_gemm_small_launch(int64_t M, int64_t N, int64_t K, const void* A, int64_t lda, const void* B, int64_t ldb, void* C,
                           int64_t ldc, const float* bias, int relu, int b_static, cudaStream_t st);
