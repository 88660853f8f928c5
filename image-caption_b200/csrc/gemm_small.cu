// Small-footprint bf16 tensor-core GEMM for the LATENCY-bound shapes of the path (decode steps: M = batch * beam rows,
// a few dozen 128 x 128 tiles per launch):   C[M,N] = act(A[M,K] . W[N,K]^T + bias)      bf16 in / bf16 out
//
// The persistent kernel of gemm_tc.cu owns a whole SM (226 KB of shared memory, all 512 TMEM columns, 320 threads x 159
// registers), so in a chain of dependent launches nothing of launch i+1 can start before the last CTA of launch i has
// left: every launch pays its own barrier init + TMEM allocation + descriptor fetch + first TMA round trip + exposed
// epilogue (measured r1: 8.4 us for a 4.8 GFLOP single-wave GEMM, of which the tensor pipe is busy ~2 us).
// This kernel is built to OVERLAP with its neighbours in the stream instead:
//   * one 128 x 128 tile per CTA, 192 threads (warp 0 TMA producer, warp 1 TMEM + MMA issuer, warps 2-5 epilogue),
//     a 3-stage 32 KB operand ring (98 KB) and 128 TMEM columns  =>  TWO CTAs per SM, of the same or of different launches;
//   * programmatic dependent launch: `griddepcontrol.launch_dependents` is issued right after the prologue, so the next
//     kernel's CTAs become resident and run THEIR prologue while this one computes; with b_static (the B operand and the
//     bias are weights that the preceding kernel does not write) the first ring stages of B are fetched BEFORE
//     `griddepcontrol.wait`, i.e. while the producer of A is still running;
//   * the epilogue stages its boxes in the (by then idle) operand ring and leaves through TMA stores.
// Replaces the reference's nn.Linear calls inside the decode loops (model.py:114-130,169-184 -> modules.py:72-77,113-114).
#include <cuda.h>
#include <stdlib.h>
#include "icap_common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 64, UMMA_K = 16;
constexpr int A_TILE_BYTES = BM * BK * 2, B_TILE_BYTES = BN * BK * 2, STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;
constexpr int NTHREADS = 192;
// STAGES = 3: 98 KB, two CTAs per SM.  STAGES = 2: 66 KB, THREE CTAs per SM -- for launches of 2..3 x #SMs tiles (decode
// FFN1: 320 tiles), which would otherwise leave a second, mostly empty wave (the SM's ingest is shared either way).
constexpr int smem_bytes(int stages) { return stages * STAGE_BYTES + 128 /*barriers*/ + BN * 4 /*bias*/ + 1024 /*align slack*/; }

struct SmallArgs {
  int M, N, K;
  const float* bias;
  int relu, b_static;
  unsigned long long* trace;     // timing experiments (icap_debug_trace): 16 globaltimer stamps of CTA (0,0), else null
};

__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

template <int STAGES>
__global__ void __launch_bounds__(NTHREADS, STAGES == 2 ? 3 : 2)
gemm_small_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmC, const SmallArgs g) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base, sB = sA + STAGES * A_TILE_BYTES, bars = sB + STAGES * B_TILE_BYTES;
  const uint32_t full_bar = bars, empty_bar = bars + 8 * STAGES, tfull_bar = bars + 16 * STAGES, slot_addr = tfull_bar + 8;
  const uint32_t sBias = bars + 128;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_raw + (slot_addr - smem_u32(smem_raw)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = (int)blockIdx.x * BN, m0 = (int)blockIdx.y * BM;
  const int nkb = (g.K + BK - 1) / BK;
  unsigned long long* const tr = (g.trace && blockIdx.x == 0 && blockIdx.y == 0) ? g.trace : nullptr;
  if (tr && threadIdx.x == 0) tr[0] = gtimer();

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmC) : "memory");
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(full_bar + 8 * i, 1);
      mbar_init(empty_bar + 8 * i, 1);
    }
    mbar_init(tfull_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_addr), "n"(BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();       // the next kernel of the stream may become resident now (it waits for OUR completion itself)
  if (tr && threadIdx.x == 0) tr[1] = gtimer();

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------ TMA producer
      const int npre = nkb < STAGES ? nkb : STAGES;
      if (g.b_static) {                      // weights: not written by the preceding kernel -> fetch before the dependency resolves
        for (int i = 0; i < npre; ++i) {
          mbar_expect_tx(full_bar + 8 * i, STAGE_BYTES);
          tma_load_2d(sB + i * B_TILE_BYTES, &tmB, i * BK, n0, full_bar + 8 * i);
        }
      }
      pdl_wait();
      if (tr) tr[2] = gtimer();
      for (int i = 0; i < npre; ++i) {
        if (!g.b_static) {
          mbar_expect_tx(full_bar + 8 * i, STAGE_BYTES);
          tma_load_2d(sB + i * B_TILE_BYTES, &tmB, i * BK, n0, full_bar + 8 * i);
        }
        tma_load_2d(sA + i * A_TILE_BYTES, &tmA, i * BK, m0, full_bar + 8 * i);
      }
      if (tr) tr[3] = gtimer();
      for (int i = npre; i < nkb; ++i) {
        const int s = i % STAGES, r = i / STAGES;
        mbar_wait(empty_bar + 8 * s, (uint32_t)((r & 1) ^ 1));
        mbar_expect_tx(full_bar + 8 * s, STAGE_BYTES);
        tma_load_2d(sA + s * A_TILE_BYTES, &tmA, i * BK, m0, full_bar + 8 * s);
        tma_load_2d(sB + s * B_TILE_BYTES, &tmB, i * BK, n0, full_bar + 8 * s);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      // ------------------------------------------------------------ MMA issuer: D=f32, A=B=bf16 K-major, 128 x 128 x 16
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % STAGES, r = i / STAGES;
        mbar_wait(full_bar + 8 * s, (uint32_t)(r & 1));
        if (tr && i == 0) tr[4] = gtimer();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t aS = sA + s * A_TILE_BYTES, bS = sB + s * B_TILE_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k)
          umma_bf16(tmem_base, make_sdesc(aS + k * 32, 16, 1024), make_sdesc(bS + k * 32, 16, 1024), idesc,
                    (i > 0 || k > 0) ? 1u : 0u);
        umma_commit(empty_bar + 8 * s);
      }
      umma_commit(tfull_bar);
      if (tr) tr[5] = gtimer();
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- epilogue warps (one TMEM lane quarter each)
    const int e = warp - 2, q = warp & 3;
    const int t128 = (int)threadIdx.x - 64;
    if (g.bias) {
      if (!g.b_static) pdl_wait();
      const float b = (n0 + t128 < g.N) ? __ldg(g.bias + n0 + t128) : 0.f;
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(sBias + (uint32_t)t128 * 4), "f"(b) : "memory");
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    mbar_wait(tfull_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tr && e == 0 && lane == 0) tr[6] = gtimer();
    const int row0 = m0 + q * 32;
    const uint32_t sw = (uint32_t)(lane & 7);
    const uint32_t ebuf = sA + (uint32_t)e * 8192u;          // two 4 KB boxes per warp, in the idle operand ring
    const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16);
    const int nchunks = min(BN / 32, (g.N - n0 + 31) / 32);
#pragma unroll
    for (int c = 0; c < BN / 32; ++c) {
      if (c < nchunks) {
        uint32_t r[32];
        tmem_ld32(tacc + (uint32_t)(c * 32), r);
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (g.bias) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 b4;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(sBias + (uint32_t)(c * 32 + j) * 4));
            v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
          }
        }
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        const uint32_t buf = ebuf + (uint32_t)(c >> 1) * 4096u, my_row = buf + (uint32_t)lane * 128u;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          uint4 o;
          __nv_bfloat162 h;
          h = __floats2bfloat162_rn(v[t * 8 + 0], v[t * 8 + 1]); o.x = *reinterpret_cast<uint32_t*>(&h);
          h = __floats2bfloat162_rn(v[t * 8 + 2], v[t * 8 + 3]); o.y = *reinterpret_cast<uint32_t*>(&h);
          h = __floats2bfloat162_rn(v[t * 8 + 4], v[t * 8 + 5]); o.z = *reinterpret_cast<uint32_t*>(&h);
          h = __floats2bfloat162_rn(v[t * 8 + 6], v[t * 8 + 7]); o.w = *reinterpret_cast<uint32_t*>(&h);
          const uint32_t addr = my_row + ((((uint32_t)((c & 1) * 4 + t)) ^ sw) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o.x), "r"(o.y), "r"(o.z), "r"(o.w) : "memory");
        }
        if ((c & 1) || c == nchunks - 1) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0 && row0 < g.M) {
            tma_store_2d(&tmC, buf, n0 + (c >> 1) * 64, row0);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    if (tr && e == 0 && lane == 0) tr[7] = gtimer();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(BN) : "memory");
  if (tr && threadIdx.x == 0) tr[8] = gtimer();
}

}  // namespace

unsigned long long* icap_g_trace = nullptr;
int icap_g_trace_slots = 0, icap_g_trace_next = 0;
unsigned long long* icap_trace_slot() {
  if (!icap_g_trace || icap_g_trace_slots <= 0) return nullptr;
  unsigned long long* p = icap_g_trace + 16 * (size_t)(icap_g_trace_next % icap_g_trace_slots);
  ++icap_g_trace_next;
  return p;
}
// timing experiments (tools/): every following tcgen05 GEMM launch writes up to 16 %globaltimer stamps of its CTA 0
// into slot (launch number % nslots) of buf (device memory, 16 x uint64 per slot); buf = NULL switches it off.
extern "C" int icap_debug_trace(unsigned long long* buf, int nslots) {
  icap_g_trace = buf;
  icap_g_trace_slots = nslots;
  icap_g_trace_next = 0;
  return 0;
}

// Is this GEMM one the small-footprint kernel takes?  (A, B K-major, bf16 out, plain store, at most ~2 co-resident waves)
bool icap_gemm_small_eligible(int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, int c_dtype, int epi,
                              int accumulate, int split_k, const void* C, int64_t ldc) {
  static IcapEnv e_mode;
  const int mode = e_mode.geti("ICAP_GEMM_SMALL", 1);     // 0 never, 1 automatic, 2 every eligible shape
  if (!mode) return false;
  if (!(a_kmajor && b_kmajor) || c_dtype != ICAP_BF16 || (epi & 15) > 1 || accumulate || split_k > 1) return false;
  if (((uintptr_t)C & 15) || (ldc % 8) || (N % 8)) return false;   // TMA stores: see icap_gemm_bf16_launch
  if (ceil_div64(M, BM) > 65535) return false;              // M tiles go on grid.y
  const int64_t tiles = ceil_div64(M, BM) * ceil_div64(N, BN);
  return tiles <= (int64_t)icap_num_sms() * 3 || mode == 2;
}

int icap_gemm_small_launch(int64_t M, int64_t N, int64_t K, const void* A, int64_t lda, const void* B, int64_t ldb, void* C,
                           int64_t ldc, const float* bias, int relu, int b_static, cudaStream_t st) {
  ICAP_ARG((uintptr_t)A % 16 == 0 && (uintptr_t)B % 16 == 0 && lda % 8 == 0 && ldb % 8 == 0,
           "icap_gemm(bf16): A/B must be 16-byte aligned with lda/ldb multiples of 8");
  CUtensorMap ta, tb, tc;
  int rc;
  if ((rc = icap_make_tmap_2d(&ta, A, M, K, lda, BM, ICAP_BF16))) return rc;
  if ((rc = icap_make_tmap_2d(&tb, B, N, K, ldb, BN, ICAP_BF16))) return rc;
  if ((rc = icap_make_tmap_2d(&tc, C, M, N, ldc, 32, ICAP_BF16))) return rc;
  static bool attr_done = false;
  if (!attr_done) {
    ICAP_CUDA(cudaFuncSetAttribute(gemm_small_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(3)));
    ICAP_CUDA(cudaFuncSetAttribute(gemm_small_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(2)));
    attr_done = true;
  }
  SmallArgs g;
  g.M = (int)M; g.N = (int)N; g.K = (int)K;
  g.bias = bias; g.relu = relu; g.b_static = b_static; g.trace = icap_trace_slot();
  const dim3 grid((unsigned)ceil_div64(N, BN), (unsigned)ceil_div64(M, BM));
  const int64_t tiles = (int64_t)grid.x * grid.y;
  static IcapEnv e_st;
  const int force = e_st.geti("ICAP_GEMM_SMALL_STAGES", 0);
  const bool two = force ? force == 2 : (tiles > 2 * (int64_t)icap_num_sms() && tiles <= 3 * (int64_t)icap_num_sms());
  if (two)
    ICAP_CUDA(icap_launch(gemm_small_kernel<2>, grid, dim3(NTHREADS), (size_t)smem_bytes(2), st, ta, tb, tc, g));
  else
    ICAP_CUDA(icap_launch(gemm_small_kernel<3>, grid, dim3(NTHREADS), (size_t)smem_bytes(3), st, ta, tb, tc, g));
  ICAP_LAUNCH_CHECK("icap_gemm(bf16, small)");
  return 0;
}
