// Tensor-core fused attention for the bf16 mode (head dim 64): one CTA per (batch, head), one warp per
// 16-query tile, mma.sync.m16n8k16 (bf16 in, fp32 accumulate) fed by ldmatrix from XOR-swizzled shared
// memory, softmax / masks / dropout in the accumulator registers with quad shuffles.
//
// The per-(b,h) problems of this model are tiny (36x36x64, 21x21x64, 21x36x64): far below the 64-row
// minimum of tcgen05.mma, so the warp-level mma.sync path is the right tensor-core instruction here; the
// large weight contractions use tcgen05 (gemm_tc.cu).
//
// Same semantics as attention.cu (ScaledDotProductAttention, modules.py:16-27): scale by 1/sqrt(dk),
// masked_fill(-inf) from key validity / causality, softmax, dropout on the probabilities, P.V.
// Backward recomputes P from Q, K (nothing is saved by the forward):
//   phase A (warp = query tile): S, P, dP = dO V^T, dS = P (dP - rowsum(P dP)); dQ = scale dS K;
//                                dS and dropped-P go to shared memory as bf16
//   phase B (warp = key tile)  : dK = scale dS^T Q ; dV = Pd^T dO
#include <stdlib.h>
#include "icap_common.cuh"

namespace {

constexpr int D = 64;             // head dim (dk == dv)
constexpr int ROWB = D * 2;       // 128 bytes per row of a [rows][64] bf16 tile

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t tile_addr(uint32_t base, int row, int chunk) {
  return base + row * ROWB + (((uint32_t)chunk ^ (uint32_t)(row & 7)) << 4);
}
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm4t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// global [rows][64] bf16 (row stride ld) -> swizzled smem tile, rows >= nrows zero-filled up to rows_pad.
// cp.async (LDGSTS, no register staging); every thread keeps its 16-byte column and steps a row pointer, so the loop
// body is one copy + one pointer add + the swizzled smem address.  Call load_tiles_wait() before the barrier.
__device__ __forceinline__ void load_tile(uint32_t sbase, const bf16* g, int64_t ld, int nrows, int rows_pad, int nthreads) {
  const int c = threadIdx.x & 7, rstep = nthreads >> 3;
  const bf16* gp = g + (int64_t)(threadIdx.x >> 3) * ld + c * 8;
  const int64_t gstep = (int64_t)rstep * ld;
  for (int r = threadIdx.x >> 3; r < rows_pad; r += rstep, gp += gstep) {
    const uint32_t dst = tile_addr(sbase, r, c);
    if (r < nrows) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gp) : "memory");
    else asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(dst), "r"(0u) : "memory");
  }
}
__device__ __forceinline__ void load_tiles_wait() {
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// bit j of word w = key 32*w + j exists and is valid (computed once per warp: NW byte loads per lane instead of one per element)
template <int NW>
__device__ __forceinline__ void key_mask(uint32_t (&km)[NW], const uint8_t* __restrict__ kvalid_b, int Lk, int lane) {
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    const int j = w * 32 + lane;
    km[w] = __ballot_sync(0xffffffffu, j < Lk && (kvalid_b == nullptr || kvalid_b[j] != 0));
  }
}

// S[16 x 8*NT8] = Q_tile K^T for this warp's query tile (rows m0..m0+15); raw dot products, fp32
template <int NT8>
__device__ __forceinline__ void qk_tile(float (&s)[NT8][4], uint32_t sQ, uint32_t sK, int m0, int lane) {
#pragma unroll
  for (int nt = 0; nt < NT8; ++nt) { s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f; }
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk) {
    uint32_t a[4];
    ldsm4(tile_addr(sQ, m0 + (lane & 15), 2 * kk + (lane >> 4)), a);
#pragma unroll
    for (int np = 0; np < NT8 / 2; ++np) {
      uint32_t b[4];
      ldsm4(tile_addr(sK, np * 16 + (lane & 7) + ((lane >> 4) << 3), 2 * kk + ((lane >> 3) & 1)), b);
      mma16816(s[2 * np], a, b[0], b[1]);
      mma16816(s[2 * np + 1], a, b[2], b[3]);
    }
  }
}

// in-register softmax over the key axis with masks; s -> normalised probabilities p (fp32).
// Thread holds rows r0 = m0 + lane/4 and r0 + 8, columns 8*nt + 2*(lane%4) + {0,1}.
template <int NT8>
__device__ __forceinline__ void softmax_tile(float (&s)[NT8][4], int m0, int lane, int Lq, int Lk, float scale,
                                             const uint8_t* __restrict__ kvalid_b, int causal) {
  constexpr int NW = (NT8 * 8 + 31) / 32;
  uint32_t km[NW];
  key_mask<NW>(km, kvalid_b, Lk, lane);
  const int r0 = m0 + (lane >> 2), r1 = r0 + 8;
  const float c = scale * 1.4426950408889634f;      // logits are kept pre-multiplied by log2(e): p = 2^(v - max)
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < NT8; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int jl = (nt & 3) * 8 + 2 * (lane & 3) + e;             // bit within word nt / 4
      const int j = nt * 8 + 2 * (lane & 3) + e;
      const bool dead = !((km[nt >> 2] >> jl) & 1u);
      const float v0 = (dead || (causal && j > r0)) ? -INFINITY : s[nt][e] * c;
      const float v1 = (dead || (causal && j > r1)) ? -INFINITY : s[nt][2 + e] * c;
      s[nt][e] = v0; s[nt][2 + e] = v1;
      mx0 = fmaxf(mx0, v0); mx1 = fmaxf(mx1, v1);
    }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < NT8; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float p0 = ex2_approx(s[nt][e] - mx0);                  // 2^(-inf) = 0 for masked keys (a fully masked
      const float p1 = ex2_approx(s[nt][2 + e] - mx1);              // row gives NaN, exactly like the reference)
      s[nt][e] = p0; s[nt][2 + e] = p1;
      sum0 += p0; sum1 += p1;
    }
  }
  sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
  sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
  const float inv0 = (r0 < Lq) ? 1.f / sum0 : 0.f, inv1 = (r1 < Lq) ? 1.f / sum1 : 0.f;   // padded query rows -> 0
#pragma unroll
  for (int nt = 0; nt < NT8; ++nt) {
    s[nt][0] *= inv0; s[nt][1] *= inv0; s[nt][2] *= inv1; s[nt][3] *= inv1;
  }
}

// keep-mask bits for this thread's elements: bit (nt*4 + e).  The element pair (row, columns 8*nt + 2*(lane%4) + {0,1})
// has pair index ((bh*Lq + row) * NT8 + nt) * 4 + lane%4, i.e. element (bh*Lq + row) * attn_drop_ld(Lk) + column
// (NT8 * 8 == attn_drop_ld(Lk) by DISPATCH_NT8) -- identical in forward and backward and in the SIMT kernels
template <int NT8>
__device__ __forceinline__ uint64_t dropout_bits(uint64_t seed, uint32_t thresh, uint64_t bh, int Lq, int m0, int lane) {
  uint64_t bits = 0;
  const int r0 = m0 + (lane >> 2);
  const uint32_t sf = seed_fold(seed);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const uint64_t base = ((bh * Lq + (uint64_t)(r0 + 8 * h)) * (uint64_t)NT8) * 4 + (uint64_t)(lane & 3);
#pragma unroll
    for (int nt = 0; nt < NT8; ++nt)
      bits |= (uint64_t)dropout_keep2(sf, base + (uint64_t)(nt * 4), thresh) << (nt * 4 + 2 * h);
  }
  return bits;
}

// out[16 x 64] = A[16 x 16*KS] (fp32 accumulator-layout registers, rounded to bf16) . B[16*KS x 64]
// with B rows = rows of a swizzled [rows][64] smem tile (transposed ldmatrix)
template <int NT8>
__device__ __forceinline__ void acc_times_tile(float (&o)[8][4], const float (&p)[NT8][4], uint32_t sB, int lane) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) { o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f; }
#pragma unroll
  for (int kk = 0; kk < NT8 / 2; ++kk) {
    uint32_t a[4];
    a[0] = pack2(p[2 * kk][0], p[2 * kk][1]);
    a[1] = pack2(p[2 * kk][2], p[2 * kk][3]);
    a[2] = pack2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
    a[3] = pack2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t b[4];
      ldsm4t(tile_addr(sB, kk * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), 2 * np + (lane >> 4)), b);
      mma16816(o[2 * np], a, b[0], b[1]);
      mma16816(o[2 * np + 1], a, b[2], b[3]);
    }
  }
}

// write a warp's [16 x 64] fp32 accumulator tile as bf16 rows m0.. of a global [rows][64] view via its own
// (already consumed) smem rows for 16-byte coalesced stores
__device__ __forceinline__ void store_tile16(const float (&o)[8][4], float mul, uint32_t sStage, int m0, int lane,
                                             bf16* g, int64_t ld, int nrows) {
  __syncwarp();
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int r = m0 + (lane >> 2);
    const uint32_t off = (uint32_t)(2 * (lane & 3)) * 2;
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(tile_addr(sStage, r, nt) + off), "r"(pack2(o[nt][0] * mul, o[nt][1] * mul)) : "memory");
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(tile_addr(sStage, r + 8, nt) + off), "r"(pack2(o[nt][2] * mul, o[nt][3] * mul)) : "memory");
  }
  __syncwarp();
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int u = it * 32 + lane, r = m0 + (u >> 3), c = u & 7;
    if (r < nrows) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(tile_addr(sStage, r, c)));
      *reinterpret_cast<uint4*>(g + (int64_t)r * ld + c * 8) = v;
    }
  }
}

template <int NT8>
__global__ void __launch_bounds__(256)
mha_fwd_mma_kernel(const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ k, int64_t ldk,
                   const bf16* __restrict__ v, int64_t ldv, bf16* __restrict__ o, int64_t ldo,
                   const uint8_t* __restrict__ kvalid, int H, int Lq, int Lk, int causal, float p_drop, uint32_t thresh,
                   uint64_t seed, const int* __restrict__ seed_dev, int kv_static) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nthreads = blockDim.x;
  const int LqP = (Lq + 15) & ~15;
  constexpr int LkP = NT8 * 8;
  const uint32_t sQ = smem_u32(smem), sK = sQ + LqP * ROWB, sV = sK + LkP * ROWB;
  // kv_static (decode cross-attention): K / V / kvalid were produced once per decode, long before this launch -- their
  // tiles are requested BEFORE the grid dependency resolves and stream in while the kernel that produces q still runs
  if (kv_static) {
    load_tile(sK, k + (int64_t)b * Lk * ldk + h * D, ldk, Lk, LkP, nthreads);
    load_tile(sV, v + (int64_t)b * Lk * ldv + h * D, ldv, Lk, LkP, nthreads);
  }
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  load_tile(sQ, q + (int64_t)b * Lq * ldq + h * D, ldq, Lq, LqP, nthreads);
  if (!kv_static) {
    load_tile(sK, k + (int64_t)b * Lk * ldk + h * D, ldk, Lk, LkP, nthreads);
    load_tile(sV, v + (int64_t)b * Lk * ldv + h * D, ldv, Lk, LkP, nthreads);
  }
  load_tiles_wait();
  __syncthreads();
  const int m0 = warp * 16;
  float s[NT8][4];
  qk_tile<NT8>(s, sQ, sK, m0, lane);
  softmax_tile<NT8>(s, m0, lane, Lq, Lk, 0.125f, kvalid ? kvalid + (int64_t)b * Lk : nullptr, causal);
  if (p_drop > 0.f) {
    const uint64_t bits = dropout_bits<NT8>(seed, thresh, (uint64_t)blockIdx.x, Lq, m0, lane);
    const float ks = 1.f / (1.f - p_drop);
#pragma unroll
    for (int nt = 0; nt < NT8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[nt][e] = ((bits >> (nt * 4 + e)) & 1) ? s[nt][e] * ks : 0.f;
  }
  float acc[8][4];
  acc_times_tile<NT8>(acc, s, sV, lane);
  store_tile16(acc, 1.f, sQ, m0, lane, o + (int64_t)b * Lq * ldo + h * D, ldo, Lq);
}

template <int NT8>
__global__ void __launch_bounds__(256)
mha_bwd_mma_kernel(const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ k, int64_t ldk,
                   const bf16* __restrict__ v, int64_t ldv, const bf16* __restrict__ dout, int64_t lddo,
                   bf16* __restrict__ dq, int64_t lddq, bf16* __restrict__ dk_, int64_t lddk, bf16* __restrict__ dv_,
                   int64_t lddv, const uint8_t* __restrict__ kvalid, int H, int Lq, int Lk, int causal, float p_drop,
                   uint32_t thresh, uint64_t seed, const int* __restrict__ seed_dev) {
  pdl_prologue();
  extern __shared__ __align__(128) uint8_t smem[];
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nthreads = blockDim.x, nwarps = nthreads >> 5;
  const int LqP = (Lq + 15) & ~15;
  constexpr int LkP = NT8 * 8;
  constexpr int SP = LkP * 2 + 16;          // row stride (bytes) of the dS / Pd tiles: odd number of 16 B chunks
  const uint32_t sQ = smem_u32(smem), sK = sQ + LqP * ROWB, sV = sK + LkP * ROWB, sDO = sV + LkP * ROWB;
  const uint32_t sDS = sDO + LqP * ROWB, sPD = sDS + LqP * SP;
  load_tile(sQ, q + (int64_t)b * Lq * ldq + h * D, ldq, Lq, LqP, nthreads);
  load_tile(sK, k + (int64_t)b * Lk * ldk + h * D, ldk, Lk, LkP, nthreads);
  load_tile(sV, v + (int64_t)b * Lk * ldv + h * D, ldv, Lk, LkP, nthreads);
  load_tile(sDO, dout + (int64_t)b * Lq * lddo + h * D, lddo, Lq, LqP, nthreads);
  load_tiles_wait();
  __syncthreads();
  const float scale = 0.125f;
  {
    // ---------------- phase A: this warp's 16 queries
    const int m0 = warp * 16;
    float p[NT8][4];
    qk_tile<NT8>(p, sQ, sK, m0, lane);
    softmax_tile<NT8>(p, m0, lane, Lq, Lk, scale, kvalid ? kvalid + (int64_t)b * Lk : nullptr, causal);
    uint64_t bits = ~0ull;
    float ks = 1.f;
    if (p_drop > 0.f) {
      bits = dropout_bits<NT8>(seed, thresh, (uint64_t)blockIdx.x, Lq, m0, lane);
      ks = 1.f / (1.f - p_drop);
    }
    // dPd = dO V^T  (same fragment layout as S)
    float dp[NT8][4];
    qk_tile<NT8>(dp, sDO, sV, m0, lane);
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT8; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool keep = (bits >> (nt * 4 + e)) & 1;
        dp[nt][e] = keep ? dp[nt][e] * ks : 0.f;             // dP
        const float t = p[nt][e] * dp[nt][e];
        if (e < 2) rs0 += t; else rs1 += t;
      }
    }
    rs0 += __shfl_xor_sync(0xffffffffu, rs0, 1); rs0 += __shfl_xor_sync(0xffffffffu, rs0, 2);
    rs1 += __shfl_xor_sync(0xffffffffu, rs1, 1); rs1 += __shfl_xor_sync(0xffffffffu, rs1, 2);
    const int r0 = m0 + (lane >> 2);
#pragma unroll
    for (int nt = 0; nt < NT8; ++nt) {
      // dropped probabilities (for dV) and dS (for dQ, dK)
      float pd[4], ds[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool keep = (bits >> (nt * 4 + e)) & 1;
        pd[e] = keep ? p[nt][e] * ks : 0.f;
        ds[e] = p[nt][e] * (dp[nt][e] - (e < 2 ? rs0 : rs1));
        dp[nt][e] = ds[e];
      }
      const uint32_t off = (uint32_t)(nt * 8 + 2 * (lane & 3)) * 2;
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sDS + r0 * SP + off), "r"(pack2(ds[0], ds[1])) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sDS + (r0 + 8) * SP + off), "r"(pack2(ds[2], ds[3])) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sPD + r0 * SP + off), "r"(pack2(pd[0], pd[1])) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sPD + (r0 + 8) * SP + off), "r"(pack2(pd[2], pd[3])) : "memory");
    }
    // dQ = scale * dS K
    float acc[8][4];
    acc_times_tile<NT8>(acc, dp, sK, lane);
    __syncthreads();      // dS / Pd are complete in shared memory; nobody reads sK / sV after this point
    // dQ stays in registers until phase B has finished reading sQ / sDO (it is staged through sDO rows)
    // ---------------- phase B: key tiles, dK = scale dS^T Q, dV = Pd^T dO
    for (int task = warp; task < 2 * (LkP / 16); task += nwarps) {
      const int jt = task >> 1, which = task & 1;      // which: 0 -> dK (dS, Q), 1 -> dV (Pd, dO)
      const uint32_t sA = which ? sPD : sDS, sB = which ? sDO : sQ;
      float out[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) { out[nt][0] = out[nt][1] = out[nt][2] = out[nt][3] = 0.f; }
      for (int kk = 0; kk < LqP / 16; ++kk) {
        uint32_t a[4];
        ldsm4t(sA + (kk * 16 + (lane & 7) + ((lane >> 4) << 3)) * SP + (uint32_t)(jt * 2 + ((lane >> 3) & 1)) * 16, a);
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          uint32_t bb[4];
          ldsm4t(tile_addr(sB, kk * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), 2 * np + (lane >> 4)), bb);
          mma16816(out[2 * np], a, bb[0], bb[1]);
          mma16816(out[2 * np + 1], a, bb[2], bb[3]);
        }
      }
      // staged through this key tile's rows of sK (dK) / sV (dV), which are dead after the barrier above
      bf16* g = which ? dv_ + (int64_t)b * Lk * lddv + h * D : dk_ + (int64_t)b * Lk * lddk + h * D;
      store_tile16(out, which ? 1.f : scale, which ? sV : sK, jt * 16, lane, g, which ? lddv : lddk, Lk);
    }
    __syncthreads();                          // phase B finished reading sQ / sDO
    store_tile16(acc, scale, sDO, m0, lane, dq + (int64_t)b * Lq * lddq + h * D, lddq, Lq);
  }
}

template <typename K>
int ensure_smem(K kern, size_t smem, size_t* cur) {
  if (smem > *cur) {
    ICAP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    *cur = smem;
  }
  return 0;
}

}  // namespace

bool icap_mha_mma_ok(int dtype, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv, int64_t ldq, int64_t ldk, int64_t ldv,
                     const void* q, const void* k, const void* v) {
  if (env_flag<3>("ICAP_MHA_SIMT")) return false;
  return dtype == ICAP_BF16 && dk == D && dv == D && Lq <= 128 && Lk <= 128 && ldq % 8 == 0 && ldk % 8 == 0 &&
         ldv % 8 == 0 && (uintptr_t)q % 16 == 0 && (uintptr_t)k % 16 == 0 && (uintptr_t)v % 16 == 0;
}

// NT8 * 8 = attn_drop_ld(Lk): the key tile of the kernel is the row stride of the dropout element index
#define DISPATCH_NT8(LK, CALL)                \
  do {                                        \
    switch (attn_drop_ld(LK)) {               \
      case 16: CALL(2); break;                \
      case 32: CALL(4); break;                \
      case 48: CALL(6); break;                \
      case 64: CALL(8); break;                \
      default: CALL(16); break;               \
    }                                         \
  } while (0)

int icap_mha_fwd_mma(int64_t B, int64_t H, int64_t Lq, int64_t Lk, const void* q, int64_t ldq, const void* k,
                     int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo, const uint8_t* kvalid, int causal,
                     float p_drop, uint64_t seed, const int* seed_dev, cudaStream_t st, int kv_static) {
  const int LqP = (int)((Lq + 15) & ~15);
  const int nthreads = 32 * (LqP / 16);
  const uint32_t th = dropout_threshold(p_drop);
#define CALL(NT)                                                                                                   \
  {                                                                                                                \
    static size_t cur = 48 * 1024;                                                                                 \
    const size_t smem = (size_t)(LqP + 2 * NT * 8) * ROWB;                                                         \
    if (int rc = ensure_smem(mha_fwd_mma_kernel<NT>, smem, &cur)) return rc;                                       \
    icap_launch(mha_fwd_mma_kernel<NT>, (unsigned)(B * H), nthreads, smem, st,                                              \
        (const bf16*)q, ldq, (const bf16*)k, ldk, (const bf16*)v, ldv, (bf16*)o, ldo, kvalid, (int)H, (int)Lq,     \
        (int)Lk, causal, p_drop, th, seed, seed_dev, kv_static);                                                   \
  }
  DISPATCH_NT8(Lk, CALL);
#undef CALL
  ICAP_LAUNCH_CHECK("icap_mha_fwd(mma)");
  return 0;
}

int icap_mha_bwd_mma(int64_t B, int64_t H, int64_t Lq, int64_t Lk, const void* q, int64_t ldq, const void* k,
                     int64_t ldk, const void* v, int64_t ldv, const void* dout, int64_t lddo, void* dq, int64_t lddq,
                     void* dk_out, int64_t lddk, void* dv_out, int64_t lddv, const uint8_t* kvalid, int causal,
                     float p_drop, uint64_t seed, const int* seed_dev, cudaStream_t st) {
  const int LqP = (int)((Lq + 15) & ~15);
  const int nthreads = 32 * (LqP / 16);
  const uint32_t th = dropout_threshold(p_drop);
#define CALL(NT)                                                                                                   \
  {                                                                                                                \
    static size_t cur = 48 * 1024;                                                                                 \
    const size_t smem = (size_t)(2 * LqP + 2 * NT * 8) * ROWB + 2 * (size_t)LqP * (NT * 16 + 16);                  \
    if (int rc = ensure_smem(mha_bwd_mma_kernel<NT>, smem, &cur)) return rc;                                       \
    icap_launch(mha_bwd_mma_kernel<NT>, (unsigned)(B * H), nthreads, smem, st,                                              \
        (const bf16*)q, ldq, (const bf16*)k, ldk, (const bf16*)v, ldv, (const bf16*)dout, lddo, (bf16*)dq, lddq,   \
        (bf16*)dk_out, lddk, (bf16*)dv_out, lddv, kvalid, (int)H, (int)Lq, (int)Lk, causal, p_drop, th, seed,      \
        seed_dev);                                                                                                 \
  }
  DISPATCH_NT8(Lk, CALL);
#undef CALL
  ICAP_LAUNCH_CHECK("icap_mha_bwd(mma)");
  return 0;
}
