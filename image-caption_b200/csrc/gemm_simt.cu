// fp32 SIMT GEMM for the fp32 parity mode (true fp32 FMA accumulation, no tensor cores).
//
//   C[M,N] (+)= op(A)[M,K] . op(B)[K,N]   (+ bias[N]) (relu | * (aux > 0))
//
// Operand storage (row-major, ld in elements):
//   a_kmajor=1 : A stored [M][K]     a_kmajor=0 : A stored [K][M]
//   b_kmajor=1 : B stored [N][K]     b_kmajor=0 : B stored [K][N]
// forward  y = x W^T          : a_kmajor=1, b_kmajor=1   (nn.Linear; modules.py:72-77)
// dgrad    dx = dy W          : a_kmajor=1, b_kmajor=0
// wgrad    dW = dy^T x        : a_kmajor=0, b_kmajor=0   (split-K, atomic accumulate)
//
// This kernel exists because the fp32 parity bar (1e-4 relative logits, identical greedy / beam
// ids) cannot be met by single-pass bf16/tf32 tensor-core math (SURVEY.md §7 "Hard parts").
#include "icap_common.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 16, PAD = 4, NT = 256;

template <bool KMAJOR>
__device__ __forceinline__ void load_tile(const float* __restrict__ P, int64_t ld, int mn0, int k0, int MN, int kend,
                                          bool vec, float (&r)[8], int tid) {
  // KMAJOR: element (mn, k) at P[mn*ld + k];  thread -> rows {tid/4, tid/4+64}, k quad (tid%4)*4
  // else  : element (mn, k) at P[k*ld + mn];  thread -> k {tid/32, tid/32+8}, mn quad (tid%32)*4
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    int mn, k;
    if (KMAJOR) { mn = mn0 + tid / 4 + i * 64; k = k0 + (tid % 4) * 4; }
    else        { k = k0 + tid / 32 + i * 8;  mn = mn0 + (tid % 32) * 4; }
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (KMAJOR) {
      if (mn < MN) {
        const float* p = P + (int64_t)mn * ld + k;
        if (vec && k + 3 < kend) v = *reinterpret_cast<const float4*>(p);
        else {
          if (k + 0 < kend) v.x = p[0];
          if (k + 1 < kend) v.y = p[1];
          if (k + 2 < kend) v.z = p[2];
          if (k + 3 < kend) v.w = p[3];
        }
      }
    } else {
      if (k < kend) {
        const float* p = P + (int64_t)k * ld + mn;
        if (vec && mn + 3 < MN) v = *reinterpret_cast<const float4*>(p);
        else {
          if (mn + 0 < MN) v.x = p[0];
          if (mn + 1 < MN) v.y = p[1];
          if (mn + 2 < MN) v.z = p[2];
          if (mn + 3 < MN) v.w = p[3];
        }
      }
    }
    r[i * 4 + 0] = v.x; r[i * 4 + 1] = v.y; r[i * 4 + 2] = v.z; r[i * 4 + 3] = v.w;
  }
}

template <bool KMAJOR>
__device__ __forceinline__ void store_tile(float (*S)[BM + PAD], const float (&r)[8], int tid) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    if (KMAJOR) {
      int mn = tid / 4 + i * 64, k = (tid % 4) * 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) S[k + j][mn] = r[i * 4 + j];
    } else {
      int k = tid / 32 + i * 8, mn = (tid % 32) * 4;
      *reinterpret_cast<float4*>(&S[k][mn]) = make_float4(r[i * 4], r[i * 4 + 1], r[i * 4 + 2], r[i * 4 + 3]);
    }
  }
}

template <bool A_KMAJOR, bool B_KMAJOR>
__global__ void __launch_bounds__(NT)
gemm_f32_kernel(int M, int N, int K, const float* __restrict__ A, int64_t lda, const float* __restrict__ B,
                int64_t ldb, float* __restrict__ C, int64_t ldc, const float* __restrict__ bias, int epi,
                const float* __restrict__ aux, int64_t ldaux, int accumulate, int kchunk, int vecA, int vecB) {
  pdl_prologue();
  __shared__ __align__(16) float As[2][BK][BM + PAD];
  __shared__ __align__(16) float Bs[2][BK][BN + PAD];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  // tiles in one grid dimension, N fastest: grid.y (at most 65535) would cap M at 8,388,480 rows
  const int tiles_n = (N + BN - 1) / BN;
  const int m0 = (int)(blockIdx.x / tiles_n) * BM, n0 = (int)(blockIdx.x % tiles_n) * BN;
  const int kbeg = blockIdx.z * kchunk, kend = min(K, kbeg + kchunk);
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float ra[8], rb[8];
  load_tile<A_KMAJOR>(A, lda, m0, kbeg, M, kend, vecA, ra, tid);
  load_tile<B_KMAJOR>(B, ldb, n0, kbeg, N, kend, vecB, rb, tid);
  store_tile<A_KMAJOR>(As[0], ra, tid);
  store_tile<B_KMAJOR>(Bs[0], rb, tid);
  __syncthreads();
  int buf = 0;
  for (int k0 = kbeg; k0 < kend; k0 += BK) {
    const bool more = (k0 + BK) < kend;
    if (more) {
      load_tile<A_KMAJOR>(A, lda, m0, k0 + BK, M, kend, vecA, ra, tid);
      load_tile<B_KMAJOR>(B, ldb, n0, k0 + BK, N, kend, vecB, rb, tid);
    }
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
      float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (more) {
      store_tile<A_KMAJOR>(As[buf ^ 1], ra, tid);
      store_tile<B_KMAJOR>(Bs[buf ^ 1], rb, tid);
      __syncthreads();
      buf ^= 1;
    }
  }

  const bool first_split = (blockIdx.z == 0);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (row >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (col >= N) continue;
      float v = acc[i][j];
      if (bias != nullptr && first_split) v += bias[col];
      if (epi == 1) v = fmaxf(v, 0.f);
      else if (epi == 2) v = (aux[(int64_t)row * ldaux + col] > 0.f) ? v : 0.f;
      float* dst = C + (int64_t)row * ldc + col;
      if (accumulate == 2) atomicAdd(dst, v);
      else if (accumulate == 1) *dst += v;
      else *dst = v;
    }
  }
}

}  // namespace

int icap_gemm_f32_launch(int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                         const float* B, int64_t ldb, float* C, int64_t ldc, const float* bias, int epi,
                         const float* aux, int64_t ldaux, int accumulate, int split_k, cudaStream_t st) {
  if (split_k < 1) split_k = 1;
  int64_t kblocks = ceil_div64(K, BK);
  if (split_k > kblocks) split_k = (int)kblocks;
  int kchunk = (int)(ceil_div64(kblocks, split_k) * BK);
  split_k = (int)ceil_div64(K, kchunk);
  if (split_k > 1) {
    ICAP_ARG(accumulate != 0 && epi == 0, "icap_gemm(fp32): split_k>1 needs accumulate!=0 and no activation epilogue");
    accumulate = 2;
  }
  int vecA = ((uintptr_t)A % 16 == 0) && (lda % 4 == 0);
  int vecB = ((uintptr_t)B % 16 == 0) && (ldb % 4 == 0);
  const int64_t tiles = ceil_div64(M, BM) * ceil_div64(N, BN);
  ICAP_ARG(tiles < (1ll << 31), "icap_gemm(fp32): %lld output tiles exceed the grid", (long long)tiles);
  dim3 grid((unsigned)tiles, 1u, (unsigned)split_k);
#define LAUNCH(AK, BKM)                                                                                            \
  icap_launch(gemm_f32_kernel<AK, BKM>, grid, NT, 0, st, (int)M, (int)N, (int)K, A, lda, B, ldb, C, ldc, bias, epi, aux, \
                                                ldaux, accumulate, kchunk, vecA, vecB)
  if (a_kmajor && b_kmajor) LAUNCH(true, true);
  else if (a_kmajor && !b_kmajor) LAUNCH(true, false);
  else if (!a_kmajor && !b_kmajor) LAUNCH(false, false);
  else LAUNCH(false, true);
#undef LAUNCH
  ICAP_LAUNCH_CHECK("icap_gemm(fp32)");
  return 0;
}
