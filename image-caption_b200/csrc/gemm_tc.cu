// bf16 tensor-core GEMM for sm_100a: TMA (cp.async.bulk.tensor) -> 128B-swizzled shared memory ->
// tcgen05.mma (cta_group::1, kind::f16, 128 x BN x 16, BN = 128 or 256) with fp32 accumulators in TMEM ->
// tcgen05.ld epilogue (bias / ReLU / ReLU-mask / accumulate / split-K reduction) -> swizzled smem -> TMA store.
//
//   C[M,N] (+)= op(A)[M,K] . op(B)[K,N]
//
// Same operand conventions as gemm_simt.cu (a_kmajor / b_kmajor); MN-major operands are fed to the
// tensor core directly through the UMMA descriptor major bits, so dgrad / wgrad need no transposes.
//
// PERSISTENT, warp-specialised (320 threads): grid = min(#tiles, #SMs), one CTA per SM (all of TMEM, ~226 KB smem).
//   warp 0      : TMA producer (one lane), 4-stage (BN=256) / 6-stage (BN=128) ring of 64-wide k-blocks
//   warp 1      : TMEM allocator + single-thread MMA issuer; TWO accumulator stages in TMEM, so the
//                 main loop of tile i+1 runs while the epilogue warps drain tile i
//   warps 2..9  : epilogue; two warps per TMEM lane quarter (warp_id % 4), each draining half of the tile's columns
//                 through its own 4 KB staging box: TMEM -> registers -> swizzled smem -> TMA store / reduce-add
// The GEMMs of this model are small (2-20 GFLOP, K = 512 mostly): per-CTA setup (barrier init, TMEM
// allocation, descriptor prefetch) is paid once per launch instead of once per tile, and the kernel is
// PDL-aware (griddepcontrol) so that setup can overlap the tail of the previous kernel in the stream.
//
// Replaces the reference's nn.Linear / torch.matmul calls (modules.py:72-77,86,113-116;
// model.py:93,295-306,433) in bf16 mode.
#include <cuda.h>
#include <stdlib.h>
#include "icap_common.cuh"
#include "tc_ptx.cuh"

namespace {

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr int BM = 128, BK = 64, UMMA_K = 16;
constexpr int A_TILE_BYTES = BM * BK * 2;        // 16 KB per stage
constexpr int NTHREADS = 320;
constexpr int EPI_WARPS = 8;                     // two per TMEM lane quarter: each takes half of the tile's columns
constexpr int EPI_BOX_BYTES = 4096;              // 32 rows x 128 B: one TMA store box
constexpr int EPI_BYTES = EPI_WARPS * EPI_BOX_BYTES;

// TWO = cta_group::2: a cluster of two CTAs (one TPC) computes a 256 x 256 tile; each CTA owns 128 rows of A and
// HALF of the B tile (128 of the 256 columns), the pair's tensor cores read both halves.  Per CTA and k-block that
// is 32 KB of operands from L2 instead of 48 KB for the same 128 x 256 x 64 MACs.
template <int BN, bool TWO> struct Cfg {
  static constexpr int B_ROWS = TWO ? BN / 2 : BN;           // B rows (n) staged per CTA
  static constexpr int B_TILE_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;
  static constexpr int STAGES = (192 * 1024) / STAGE_BYTES;  // 4 (128x256), 6 (128x128 and 2-CTA)
  static constexpr int TMEM_COLS = 2 * BN;                   // two accumulator stages
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 256 /*barriers*/ + 1024 /*bias staging*/ +
                                    1024 /*align slack*/;
};


// 32 consecutive elements of the ReLU-mask operand (aux) of one row, as raw 16-byte words
template <typename TO> struct AuxRow { uint4 w[32 * sizeof(TO) / 16]; };
template <typename TO>
__device__ __forceinline__ void aux_load(AuxRow<TO>& a, const TO* __restrict__ p, bool vec, int ncols) {
  constexpr int NW = 32 * sizeof(TO) / 16, EPW = 16 / sizeof(TO);
  if (vec) {
#pragma unroll
    for (int t = 0; t < NW; ++t) a.w[t] = __ldg(reinterpret_cast<const uint4*>(p) + t);
  } else {
    TO* e = reinterpret_cast<TO*>(a.w);
#pragma unroll
    for (int j = 0; j < NW * EPW; ++j) e[j] = j < ncols ? p[j] : from_f32<TO>(0.f);
  }
}
template <typename TO>
__device__ __forceinline__ void aux_mask(const AuxRow<TO>& a, float (&v)[32]) {
  const TO* e = reinterpret_cast<const TO*>(a.w);
#pragma unroll
  for (int j = 0; j < 32; ++j) if (!(to_f32(e[j]) > 0.f)) v[j] = 0.f;
}

struct GemmArgs {
  int M, N, K;
  void* C;
  int64_t ldc;
  const float* bias;
  int epi;
  const void* aux;
  int64_t ldaux;
  int accumulate;      // 0 store, 1 C += (load/add/store or TMA reduce), 2 atomics (split-K on the direct path)
  int kb_per_split, splits, tiles_m, tiles_n;
  int vec_ok, store_mode;   // store_mode: 0 direct global stores, 1 TMA store, 2 TMA reduce-add
  int debug;                // timing experiments only (ICAP_GEMM_DEBUG): 1 = no TMA loads, 2 = no MMAs, 3 = no epilogue stores
  unsigned long long* trace; // timing experiments (icap_debug_trace): %globaltimer stamps of CTA 0, else null
  int b_static;             // B / bias are weights the preceding kernel does not write: fetch B before griddepcontrol.wait
};

__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

template <int BN, bool TWO, bool A_KMAJOR, bool B_KMAJOR, typename TO, bool STATS = false>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const GemmArgs g) {
  using CF = Cfg<BN, TWO>;
  constexpr int STAGES = CF::STAGES;
  constexpr int NCTA = TWO ? 2 : 1;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base, sB = sA + STAGES * A_TILE_BYTES, sE = sB + STAGES * CF::B_TILE_BYTES;
  const uint32_t bars = sE + EPI_BYTES;                  // full[S], empty[S], tfull[2], tempty[2], tmem slot
  const uint32_t full_bar = bars, empty_bar = bars + 8 * STAGES, tfull_bar = bars + 16 * STAGES;
  const uint32_t tempty_bar = tfull_bar + 16, slot_addr = tempty_bar + 16;
  const uint32_t sBias = bars + 256;                     // 8 x 128 B: one 32-float bias row per epilogue warp
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_raw + (slot_addr - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int M = g.M, N = g.N;
  const int nkb_total = (g.K + BK - 1) / BK;
  const int total_tiles = g.tiles_m * g.tiles_n * g.splits;      // tiles of (NCTA*128) x BN
  const uint32_t rank = TWO ? cluster_ctarank() : 0u;            // 0 = leader of the pair
  const int worker = TWO ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int nworkers = TWO ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  unsigned long long* const tr = (g.trace && blockIdx.x == 0) ? g.trace : nullptr;
  if (tr && threadIdx.x == 0) tr[0] = gtimer();

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    if (g.store_mode) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmC) : "memory");
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(full_bar + 8 * i, 1);                    // pair: only the leader arrives (expect_tx of BOTH CTAs' bytes)
      mbar_init(empty_bar + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar + 8 * i, 1);
      mbar_init(tempty_bar + 8 * i, EPI_WARPS * NCTA);   // pair: the peer's epilogue warps arrive remotely
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (TWO) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_addr), "n"(CF::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_addr), "n"(CF::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if constexpr (TWO) cluster_sync_all(); else __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  if (tr && threadIdx.x == 0) tr[1] = gtimer();
  // PDL: everything above overlaps the previous kernel's tail.  The next kernel of the stream may become resident from
  // here on (it waits for OUR completion itself); our own grid dependency is resolved by the TMA producer -- with
  // b_static only after it has requested the B (weight) tiles of its first ring round -- and by the epilogue warps
  // before they touch C / aux.
  pdl_launch_dependents();
  if (warp != 0) pdl_wait();
  if (tr && threadIdx.x == 0) tr[2] = gtimer();

  if (warp == 0) {
    if (lane == 0) {
      // ------------------------------------------------------------ TMA producer (one per CTA)
      const uint32_t full_leader = TWO ? map_to_cta(full_bar, 0) : full_bar;
      int s = 0, ph = 0;
      // b_static (single-CTA tiles): the B tiles of the first ring round of this CTA's first tile are requested before
      // the grid dependency resolves; `pre_b` stages already carry their expect_tx and their B bytes
      int pre_b = 0;
      if constexpr (!TWO) {
        if (g.b_static && (g.debug & 7) != 1 && worker < total_tiles) {
          const int n0 = (worker % g.tiles_n) * BN;
          const int kb0 = (worker / (g.tiles_n * g.tiles_m)) * g.kb_per_split;
          const int nkb = min(g.kb_per_split, nkb_total - kb0);
          pre_b = min(nkb, STAGES);
          for (int i = 0; i < pre_b; ++i) {
            const int k0 = (kb0 + i) * BK;
            const uint32_t dB = sB + i * CF::B_TILE_BYTES;
            mbar_expect_tx(full_bar + 8 * i, CF::STAGE_BYTES);
            if (B_KMAJOR) tma_load_2d(dB, &tmB, k0, n0, full_bar + 8 * i);
            else {
#pragma unroll
              for (int j = 0; j < BN / 64; ++j) tma_load_2d(dB + j * 8192, &tmB, n0 + 64 * j, k0, full_bar + 8 * i);
            }
          }
        }
      }
      pdl_wait();
      for (int tile = worker; tile < total_tiles; tile += nworkers) {
        const int n0 = (tile % g.tiles_n) * BN + (int)rank * CF::B_ROWS;       // this CTA's share of the B tile
        const int m0 = ((tile / g.tiles_n) % g.tiles_m) * (BM * NCTA) + (int)rank * BM;
        const int kb0 = (tile / (g.tiles_n * g.tiles_m)) * g.kb_per_split;
        const int nkb = min(g.kb_per_split, nkb_total - kb0);
        for (int i = 0; i < nkb; ++i) {
          const int k0 = (kb0 + i) * BK;
          const uint32_t dA = sA + s * A_TILE_BYTES, dB = sB + s * CF::B_TILE_BYTES;
          if (pre_b > 0) {                       // first ring round of the first tile: B is already on its way
            --pre_b;
            if (A_KMAJOR) tma_load_2d(dA, &tmA, k0, m0, full_bar + 8 * s);
            else {
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) tma_load_2d(dA + j * 8192, &tmA, m0 + 64 * j, k0, full_bar + 8 * s);
            }
            if (++s == STAGES) { s = 0; ph ^= 1; }
            continue;
          }
          mbar_wait_t<TWO>(empty_bar + 8 * s, ph ^ 1);
          if ((g.debug & 7) == 1) {                    // timing experiment: barriers only, operands are garbage
            if (rank == 0) mbar_arrive(full_bar + 8 * s);
          } else if constexpr (TWO) {
            const uint32_t fb = full_leader + 8 * s;
            // Both CTAs' TMA bytes complete on the leader's barrier.  The peer does NOT arrive on it: a remote
            // mbarrier.arrive.release.cluster per k-block cost ~0.5 us each (measured, tools/gemm_bench.py).
            if (rank == 0) mbar_expect_tx(full_bar + 8 * s, 2 * CF::STAGE_BYTES);
            if (A_KMAJOR) tma_load_2d_2sm(dA, &tmA, k0, m0, fb);
            else {
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) tma_load_2d_2sm(dA + j * 8192, &tmA, m0 + 64 * j, k0, fb);
            }
            if (B_KMAJOR) tma_load_2d_2sm(dB, &tmB, k0, n0, fb);                    // box {64 k, 128 n}
            else {
#pragma unroll
              for (int j = 0; j < CF::B_ROWS / 64; ++j) tma_load_2d_2sm(dB + j * 8192, &tmB, n0 + 64 * j, k0, fb);
            }
          } else {
            mbar_expect_tx(full_bar + 8 * s, CF::STAGE_BYTES);
            if (A_KMAJOR) tma_load_2d(dA, &tmA, k0, m0, full_bar + 8 * s);          // box {64 k, 128 m}
            else {                                                                   // 2 boxes {64 m, 64 k}
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) tma_load_2d(dA + j * 8192, &tmA, m0 + 64 * j, k0, full_bar + 8 * s);
            }
            if (B_KMAJOR) tma_load_2d(dB, &tmB, k0, n0, full_bar + 8 * s);          // box {64 k, BN n}
            else {
#pragma unroll
              for (int j = 0; j < BN / 64; ++j) tma_load_2d(dB + j * 8192, &tmB, n0 + 64 * j, k0, full_bar + 8 * s);
            }
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      // ------------------------------------------------------------ MMA issuer (one thread; pair: leader CTA only)
      // instruction descriptor: D=f32, A=B=bf16, majors, N>>3, M>>4   (pair: M = 256 across the two CTAs)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_KMAJOR ? 0u : 1u) << 15) |
                             ((B_KMAJOR ? 0u : 1u) << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)((BM * NCTA) >> 4) << 24);
      int s = 0, ph = 0, it = 0;
      for (int tile = worker; tile < total_tiles; tile += nworkers, ++it) {
        const int kb0 = (tile / (g.tiles_n * g.tiles_m)) * g.kb_per_split;
        const int nkb = min(g.kb_per_split, nkb_total - kb0);
        const int as = it & 1, aph = (it >> 1) & 1;
        mbar_wait_t<TWO>(tempty_bar + 8 * as, aph ^ 1);          // epilogue has drained this accumulator stage
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tacc = tmem_base + (uint32_t)(as * BN);
        for (int i = 0; i < nkb; ++i) {
          mbar_wait_t<TWO>(full_bar + 8 * s, ph);
          if (tr && it == 0 && i == 0) tr[4] = gtimer();
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t aS = sA + s * A_TILE_BYTES, bS = sB + s * CF::B_TILE_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // K-major : 8-row groups 1024 B apart (SBO), +32 B per 16-element k step inside the swizzle atom
            // MN-major: 64-element MN atoms 8192 B apart (LBO), 8-k groups 1024 B apart (SBO), +2048 B per k step
            const uint64_t ad = A_KMAJOR ? make_sdesc(aS + k * 32, 16, 1024) : make_sdesc(aS + k * 2048, 8192, 1024);
            const uint64_t bd = B_KMAJOR ? make_sdesc(bS + k * 32, 16, 1024) : make_sdesc(bS + k * 2048, 8192, 1024);
            if ((g.debug & 7) == 2) continue;
            if constexpr (TWO) umma_bf16_2sm(tacc, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
            else umma_bf16(tacc, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
          }
          // smem slot free (in both CTAs of a pair) once these MMAs have read it
          if constexpr (TWO) umma_commit_2sm(empty_bar + 8 * s); else umma_commit(empty_bar + 8 * s);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        // accumulator complete
        if constexpr (TWO) umma_commit_2sm(tfull_bar + 8 * as); else umma_commit(tfull_bar + 8 * as);
        if (tr && it == 0) tr[5] = gtimer();
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue warps
    constexpr int ESZ = (int)sizeof(TO);
    constexpr int CPB = 128 / ESZ;             // columns per TMA store box (one 128 B swizzle row): 64 bf16 / 32 fp32
    constexpr int CHUNKS_PER_BOX = CPB / 32;   // 32-column TMEM loads per box
    constexpr int NCH = 32 * ESZ / 16;         // 16 B smem chunks per 32 columns: 4 (bf16) / 8 (fp32)
    // The epilogue is one dependent instruction stream per warp (TMEM load -> math -> convert -> st.shared), i.e.
    // latency bound: with 4 warps it took ~3.7 us per 128x256 tile, longer than a K=512 main loop (ncu/ablation r1).
    // Eight warps -- two per TMEM lane quarter, each draining half of the columns -- halve that.
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int ew = warp - 2, half = ew >> 2;   // half: which half of the tile's columns
    const uint32_t ebuf = sE + (uint32_t)ew * EPI_BOX_BYTES;
    const uint32_t sw = (uint32_t)(lane & 7);
    TO* const C = reinterpret_cast<TO*>(g.C);
    const TO* const aux = reinterpret_cast<const TO*>(g.aux);
    const uint32_t tempty_leader = TWO ? map_to_cta(tempty_bar, 0) : tempty_bar;
    int it = 0, nbox = 0;
    for (int tile = worker; tile < total_tiles; tile += nworkers, ++it) {
      const int n0 = (tile % g.tiles_n) * BN;
      const int m0 = ((tile / g.tiles_n) % g.tiles_m) * (BM * NCTA) + (int)rank * BM;
      const bool add_bias = (g.bias != nullptr) && (tile < g.tiles_n * g.tiles_m);     // split 0 only
      const int as = it & 1, aph = (it >> 1) & 1;
      const int row0 = m0 + q * 32, row = row0 + lane;
      const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);
      const int c_begin = half * (BN / 64);
      const int nchunks = min((half + 1) * (BN / 64), (N - n0 + 31) / 32);      // this warp: chunks [c_begin, nchunks)
      AuxRow<TO> a_cur, a_nxt;
      const bool aux_vec = g.vec_ok != 0;
      // epi == 3 (classifier -> beam select): running (largest, second largest, sum of exp(x - largest)) of this thread's
      // row over this warp's columns of the tile, on the ROUNDED values that are stored
      float st_m1 = -INFINITY, st_m2 = -INFINITY, st_s = 0.f;
      if (g.epi == 2 && row < M && c_begin < nchunks)
        aux_load(a_cur, aux + (int64_t)row * g.ldaux + n0 + c_begin * 32, aux_vec && n0 + c_begin * 32 + 32 <= N,
                 N - n0 - c_begin * 32);
      mbar_wait_t<TWO>(tfull_bar + 8 * as, aph);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (tr && it == 0 && ew == 0 && lane == 0) tr[6] = gtimer();
      if (c_begin >= nchunks) {                 // ragged N: nothing to drain, just hand the stage back
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          if constexpr (TWO) mbar_arrive_cluster(tempty_leader + 8 * as); else mbar_arrive(tempty_bar + 8 * as);
        }
      }
#pragma unroll 1
      for (int c = c_begin; c < nchunks; ++c) {
        const int col0 = n0 + c * 32;
        if (g.epi == 2 && row < M && c + 1 < nchunks)
          aux_load(a_nxt, aux + (int64_t)row * g.ldaux + col0 + 32, aux_vec && col0 + 64 <= N, N - col0 - 32);
        float bias_l = 0.f;                     // lane j holds bias[col0 + j]; broadcast through smem below
        if (add_bias && col0 + lane < N) bias_l = __ldg(g.bias + col0 + lane);
        uint32_t r[32];
        tmem_ld32(tacc + (uint32_t)(c * 32), r);
        if (c == nchunks - 1) {                 // accumulator fully read: hand the TMEM stage back to the MMA warp
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            if constexpr (TWO) mbar_arrive_cluster(tempty_leader + 8 * as); else mbar_arrive(tempty_bar + 8 * as);
          }
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (add_bias) {
          const uint32_t bslot = sBias + (uint32_t)ew * 128;
          __syncwarp();                         // previous chunk's reads of the slot are done
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(bslot + (uint32_t)lane * 4), "f"(bias_l) : "memory");
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 b4;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(bslot + (uint32_t)j * 4));
            v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
          }
        }
        if (g.epi == 1) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        } else if (g.epi == 2) {
          if (row < M) aux_mask<TO>(a_cur, v);
          a_cur = a_nxt;
        }
        if constexpr (STATS) {
          {
            // The epilogue warps have two warps per scheduler: dependent chains cost their full latency.  So: top-2 on
            // PACKED bf16 pairs in two independent chains (3 instructions per two logits), the exp-sum in four
            // accumulators, the bf16 rounding shared with the store below (same cvt, merged by the compiler).
            uint32_t pk[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
              pk[j] = *reinterpret_cast<const uint32_t*>(&h);
            }
            if (col0 + 32 > N) {                       // ragged last chunk of the row: columns >= N count as -inf
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                if (col0 + 2 * j >= N) pk[j] = (pk[j] & 0xffff0000u) | 0xff80u;
                if (col0 + 2 * j + 1 >= N) pk[j] = (pk[j] & 0xffffu) | 0xff800000u;
              }
            }
            const uint32_t ninf2 = 0xff80ff80u;
            __nv_bfloat162 a1 = *reinterpret_cast<const __nv_bfloat162*>(&ninf2), a2 = a1, b1 = a1, b2 = a1;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const __nv_bfloat162 wa = *reinterpret_cast<const __nv_bfloat162*>(&pk[j]);
              const __nv_bfloat162 wb = *reinterpret_cast<const __nv_bfloat162*>(&pk[8 + j]);
              a2 = __hmax2(a2, __hmin2(a1, wa)); a1 = __hmax2(a1, wa);
              b2 = __hmax2(b2, __hmin2(b1, wb)); b1 = __hmax2(b1, wb);
            }
            const __nv_bfloat162 p1 = __hmax2(a1, b1), p2 = __hmax2(__hmin2(a1, b1), __hmax2(a2, b2));
            const float l1 = __low2float(p1), h1 = __high2float(p1), l2 = __low2float(p2), h2 = __high2float(p2);
            const float cm1 = fmaxf(l1, h1), cm2 = fmaxf(fminf(l1, h1), fmaxf(l2, h2));
            const float mn = fmaxf(st_m1, cm1);
            if (mn > -INFINITY) {
              constexpr float LOG2E = 1.4426950408889634f;
              const float nb = -mn * LOG2E;
              float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                s4[(2 * j) & 3] += ex2_approx(fmaf(__uint_as_float(pk[j] << 16), LOG2E, nb));
                s4[(2 * j + 1) & 3] += ex2_approx(fmaf(__uint_as_float(pk[j] & 0xffff0000u), LOG2E, nb));
              }
              st_s = st_s * ex2_approx((st_m1 - mn) * LOG2E) + ((s4[0] + s4[1]) + (s4[2] + s4[3]));
            }
            st_m2 = fmaxf(fmaxf(st_m2, cm2), fminf(st_m1, cm1));
            st_m1 = mn;
          }
        }
        if ((g.debug & 7) == 3) {                     // timing experiment: no stores at all (keep the math alive)
          float acc = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) acc += v[j];
          if (acc == 123.456f) C[0] = from_f32<TO>(acc);
        } else if (g.store_mode != 0) {
          // ---- staged: registers -> 128B-swizzled smem box (32 rows x 128 B) -> TMA store / reduce-add
          const int cc = c % CHUNKS_PER_BOX;
          const uint32_t buf = ebuf;
          if (cc == 0) {                        // the TMA store that last read this buffer must be done
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            __syncwarp();
          }
          const uint32_t my_row = buf + (uint32_t)lane * 128;
#pragma unroll
          for (int t = 0; t < NCH; ++t) {
            const uint32_t addr = my_row + ((((uint32_t)(cc * NCH + t)) ^ sw) << 4);
            uint4 o;
            if constexpr (ESZ == 2) {
              __nv_bfloat162 h;
              h = __floats2bfloat162_rn(v[t * 8 + 0], v[t * 8 + 1]); o.x = *reinterpret_cast<uint32_t*>(&h);
              h = __floats2bfloat162_rn(v[t * 8 + 2], v[t * 8 + 3]); o.y = *reinterpret_cast<uint32_t*>(&h);
              h = __floats2bfloat162_rn(v[t * 8 + 4], v[t * 8 + 5]); o.z = *reinterpret_cast<uint32_t*>(&h);
              h = __floats2bfloat162_rn(v[t * 8 + 6], v[t * 8 + 7]); o.w = *reinterpret_cast<uint32_t*>(&h);
            } else {
              o.x = __float_as_uint(v[t * 4 + 0]); o.y = __float_as_uint(v[t * 4 + 1]);
              o.z = __float_as_uint(v[t * 4 + 2]); o.w = __float_as_uint(v[t * 4 + 3]);
            }
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o.x), "r"(o.y), "r"(o.z), "r"(o.w) : "memory");
          }
          if (cc == CHUNKS_PER_BOX - 1 || c == nchunks - 1) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
              if (row0 < M) {
                const int bc0 = n0 + (c / CHUNKS_PER_BOX) * CPB;
                if (g.store_mode == 2) tma_reduce_add_2d(&tmC, buf, bc0, row0);
                else tma_store_2d(&tmC, buf, bc0, row0);
              }
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            ++nbox;
          }
        } else if (row < M) {
          // ---- direct global stores (C not TMA-aligned)
          TO* crow = C + (int64_t)row * g.ldc + col0;
          const bool full = g.vec_ok && (col0 + 32 <= N);
          if (g.accumulate == 2) {
            if constexpr (sizeof(TO) == 4) {
              for (int j = 0; j < 32; ++j) if (col0 + j < N) atomicAdd(reinterpret_cast<float*>(crow) + j, v[j]);
            }
          } else if (full) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              if (g.accumulate == 1) {      // C + round(v), as the TMA reduce-add of the staged path computes it
                float o[8];
                OutVec<TO>::load8(crow + j, o);
#pragma unroll
                for (int t = 0; t < 8; ++t) v[j + t] = to_f32(from_f32<TO>(v[j + t])) + o[t];
              }
              OutVec<TO>::store8(crow + j, v + j);
            }
          } else {
            for (int j = 0; j < 32; ++j) {
              if (col0 + j < N) {
                float o = v[j];
                if (g.accumulate == 1) o = to_f32(from_f32<TO>(o)) + to_f32(crow[j]);
                crow[j] = from_f32<TO>(o);
              }
            }
          }
        }
      }
      if (STATS && row < M) {
        float* sp = const_cast<float*>(reinterpret_cast<const float*>(g.aux)) + (int64_t)row * g.ldaux +
                    (int64_t)((tile % g.tiles_n) * 2 + half) * 4;
        *reinterpret_cast<float4*>(sp) = make_float4(st_m1, st_m2, st_s, 0.f);
      }
    }
    if (g.store_mode != 0 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (tr && ew == 0 && lane == 0) tr[7] = gtimer();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if constexpr (TWO) cluster_sync_all(); else __syncthreads();    // pair: the peer may still signal our barriers / read our smem
  if (warp == 1) {
    if constexpr (TWO)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(CF::TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(CF::TMEM_COLS) : "memory");
  }
  if (tr && threadIdx.x == 0) tr[8] = gtimer();
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D row-major tensor [rows][cols] (ld elements) with a 128-byte-wide box of box_rows rows, 128B swizzle
int make_tmap(CUtensorMap* tm, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows,
              int dtype = ICAP_BF16) {
  EncodeTiledFn fn = get_encode_fn();
  ICAP_ARG(fn != nullptr, "cuTensorMapEncodeTiled entry point not found (driver too old?)");
  const int esz = dtype == ICAP_BF16 ? 2 : 4;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  static IcapEnv e_promo;
  const int promo_env = e_promo.geti("ICAP_TMA_L2_PROMOTION", 256);
  const CUtensorMapL2promotion promo = promo_env == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE
                                       : promo_env == 64 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                       : promo_env == 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                                                          : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
  CUresult r = fn(tm, dtype == ICAP_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                  const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  ICAP_ARG(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d): ptr=%p rows=%lld cols=%lld ld=%lld", (int)r, ptr,
           (long long)rows, (long long)cols, (long long)ld);
  return 0;
}

int g_num_sms = 0, g_num_sms_gen = -1, g_sms_limit = 0;

int num_sms_all();
int num_sms() {
  const int n = num_sms_all();
  return (g_sms_limit > 0 && g_sms_limit < n) ? g_sms_limit : n;
}
int num_sms_all() {
  if (g_num_sms == 0 || g_num_sms_gen != icap_g_env_gen) {
    g_num_sms_gen = icap_g_env_gen;
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      g_num_sms = n;
    else
      g_num_sms = 148;
    if (const char* e = getenv("ICAP_GEMM_SMS")) { int v = atoi(e); if (v > 0) g_num_sms = v; }   // once per env generation
  }
  return g_num_sms;
}

template <int BN, bool TWO, bool AK, bool BKM, typename TO, bool STATS = false>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& g, cudaStream_t st) {
  static bool attr_done = false;
  auto kern = gemm_tc_kernel<BN, TWO, AK, BKM, TO, STATS>;
  using CF = Cfg<BN, TWO>;
  if (!attr_done) {
    ICAP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CF::SMEM_BYTES));
    attr_done = true;
  }
  const int total = g.tiles_m * g.tiles_n * g.splits;
  if (!TWO) {
    ICAP_CUDA(icap_launch(kern, dim3((unsigned)(total < num_sms() ? total : num_sms())), dim3(NTHREADS),
                          (size_t)CF::SMEM_BYTES, st, ta, tb, tc, g));
    return 0;
  }
  // CTA pairs: cluster (2,1,1), one pair per TPC, persistent over the 256 x BN tiles
  const int pairs = num_sms() / 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * (total < pairs ? total : pairs)));
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = CF::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = icap_g_pdl ? 2 : 1;
  ICAP_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, g));
  return 0;
}

// Estimated tensor-pipe clocks of the whole launch (persistent: waves x per-tile main loop, plus one exposed
// epilogue); picks the tile configuration and the split-K factor.  cfg: 0 = 128x128, 1 = 128x256, 2 = CTA pair 256x256.
// Per-k-block costs are calibrated with tools/gemm_bench.py: the main loop is bound by operand bytes from L2
// (128x128: 32 KB per 128x128x64 MACs; 128x256: 48 KB per 2x that; pair: 32 KB per CTA per 2x that).
double est_cost(int64_t tiles, int nkb, int cfg, int sms) {
  const int workers = cfg == 2 ? sms / 2 : sms;
  const double waves = (double)((tiles + workers - 1) / workers);
  const double per_kb = cfg == 0 ? 345.0 : cfg == 1 ? 512.0 : 400.0;
  const double epi = cfg == 0 ? 512.0 : 1024.0;
  return waves * (double)nkb * per_kb + epi + (cfg == 2 ? 2200.0 : 1500.0);
}

}  // namespace

int icap_make_tmap_2d(CUtensorMap* tm, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, int dtype) {
  return make_tmap(tm, ptr, rows, cols, ld, box_rows, dtype);
}
int icap_num_sms() { return num_sms(); }
// Persistent-grid width of the following icap_gemm(bf16) launches (0 = every SM).  Data parallel: the backward leaves
// a few SMs to the NCCL all-reduce kernels that run beside it (a 226 KB-smem GEMM CTA cannot share its SM with them).
extern "C" int icap_set_gemm_sms(int n) { g_sms_limit = n; return 0; }

int icap_gemm_bf16_launch(int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda,
                          const void* B, int64_t ldb, void* C, int64_t ldc, int c_dtype, const float* bias, int epi,
                          const void* aux, int64_t ldaux, int accumulate, int split_k, cudaStream_t st) {
  ICAP_ARG((uintptr_t)A % 16 == 0 && (uintptr_t)B % 16 == 0, "icap_gemm(bf16): A/B must be 16-byte aligned");
  // latency-bound shapes (decode steps): the small-footprint kernel that overlaps with its neighbours in the stream
  if (icap_gemm_small_eligible(a_kmajor, b_kmajor, M, N, K, c_dtype, epi, accumulate, split_k, C, ldc))
    return icap_gemm_small_launch(M, N, K, A, lda, B, ldb, C, ldc, bias, (epi & 15) == 1, (epi & 16) != 0, st);
  static IcapEnv e_nopre;
  const int b_static = ((epi & 16) != 0 && !e_nopre.get("ICAP_GEMM_NO_B_PREFETCH")) ? 1 : 0;
  epi &= 15;
  ICAP_ARG(lda % 8 == 0 && ldb % 8 == 0, "icap_gemm(bf16): lda/ldb must be multiples of 8 (TMA 16-byte strides)");
  ICAP_ARG(!(a_kmajor == 0 && b_kmajor == 1), "icap_gemm(bf16): (A MN-major, B K-major) is not instantiated");
  const int sms = num_sms();
  const int nkb = (int)ceil_div64(K, BK);
  const bool can_split = accumulate != 0 && epi == 0 && c_dtype == ICAP_F32 && bias == nullptr;
  // ---- tile configuration and split-K factor: split_k <= 0 = automatic (fill the SMs, >= 4 k-blocks per split)
  int best_cfg = 0, best_split = 1;
  double best_cost = 1e30;
  static IcapEnv e_bn, e_nopair, e_direct, e_dbg;
  const char* force_bn = e_bn.get("ICAP_GEMM_BN");                     // "128" | "256" | "pair"
  const bool no_pair = e_nopair.get("ICAP_GEMM_NO_PAIR") != nullptr;
  const bool direct_epi = e_direct.get("ICAP_GEMM_DIRECT_EPILOGUE") != nullptr;
  const bool pair_ok = sms >= 2;               // a CTA pair occupies two SMs: a one-SM grid runs 128x128 tiles instead
  for (int c = 2; c >= 0; --c) {
    if (force_bn && epi != 3) {
      const int want = force_bn[0] == 'p' ? (pair_ok ? 2 : 0) : (atoi(force_bn) == 256 ? 1 : 0);
      if (want != c) continue;
    }
    const int bn = c == 0 ? 128 : 256, bm = c == 2 ? 256 : 128;
    if (epi == 3 && c != 1) continue;          // row statistics: one partial per 128 columns = per column half of a 128x256 tile
    if (c >= 1 && N <= 128 && !force_bn && epi != 3) continue;
    if (c == 2 && (!pair_ok || (!force_bn && (M <= 128 || no_pair)))) continue;
    const int64_t tiles = ceil_div64(M, bm) * ceil_div64(N, bn);
    const int workers = c == 2 ? sms / 2 : sms;
    int split = split_k;
    if (split <= 0) {
      split = 1;
      if (can_split && tiles < workers) {
        split = (int)(workers / tiles);
        if (split > nkb / 4) split = nkb / 4;
        if (split < 1) split = 1;
      }
    }
    if (split > nkb) split = nkb;
    if (split > 1 && !can_split) split = 1;
    int kb_per = (nkb + split - 1) / split;
    split = (nkb + kb_per - 1) / kb_per;
    double cost = est_cost(tiles * split, kb_per, c, sms);
    if (c == 2 && !force_bn) {
      // CTA pairs (2/3 of the operand traffic, ~1 us more setup) only pay off for long per-worker k loops, or when
      // an operand's row pitch is not a multiple of 128 B (every TMA box row then straddles two L2 lines):
      // measured with tools/gemm_bench.py -- embed / classifier dgrad+wgrad win 12-18 %, K <= 2048 shapes lose ~10 %.
      const int64_t work = (int64_t)kb_per * ((tiles * split + workers - 1) / workers);
      const bool ragged_pitch = (lda * 2) % 128 != 0 || (ldb * 2) % 128 != 0;
      if (!(work >= 80 || (ragged_pitch && work >= 32))) continue;
      cost = 0.0;                            // eligible: take it
    }
    if (cost < best_cost) { best_cost = cost; best_cfg = c; best_split = split; }
  }
  if (epi == 3) {
    ICAP_ARG(c_dtype == ICAP_BF16 && !accumulate && split_k <= 1 && aux && ((uintptr_t)aux & 15) == 0 &&
             ldaux >= 8 * ceil_div64(N, 256) && ldaux % 4 == 0 && best_cfg == 1 && a_kmajor && b_kmajor,
             "icap_gemm(bf16): the row-statistics epilogue needs K-major A and B, bf16 C, no accumulation and a 16-byte "
             "aligned stats buffer of >= 8 * ceil(N / 256) floats per row");
  }
  if (split_k > 1)
    ICAP_ARG(can_split, "icap_gemm(bf16): split_k>1 needs fp32 C, accumulate!=0, no bias and no activation epilogue");
  split_k = best_split;
  const bool two = best_cfg == 2;
  const int BN = best_cfg == 0 ? 128 : 256;
  const int kb_per = (nkb + split_k - 1) / split_k;
  if (split_k > 1) accumulate = 2;
  ICAP_ARG(accumulate != 2 || c_dtype == ICAP_F32, "icap_gemm(bf16): atomic accumulate needs fp32 C");

  CUtensorMap ta, tb;
  int rc;
  if (a_kmajor) rc = make_tmap(&ta, A, M, K, lda, BM); else rc = make_tmap(&ta, A, K, M, lda, 64);
  if (rc) return rc;
  if (b_kmajor) rc = make_tmap(&tb, B, N, K, ldb, two ? BN / 2 : BN); else rc = make_tmap(&tb, B, K, N, ldb, 64);
  if (rc) return rc;
  const int esz = c_dtype == ICAP_F32 ? 4 : 2;
  int vec_ok = ((uintptr_t)C % 16 == 0) && ((ldc * esz) % 16 == 0);
  // staged TMA epilogue whenever C satisfies the TMA alignment rules and its rows end on a 16-byte boundary (a TMA
  // store / reduce-add of a row ending inside a 16-byte chunk also writes the rest of that chunk, past N: observed on
  // B200); accumulation = TMA reduce-add
  int store_mode = vec_ok && (N * esz) % 16 == 0 ? (accumulate ? 2 : 1) : 0;
  if (direct_epi) store_mode = 0;
  if (epi == 2) vec_ok = vec_ok && ((uintptr_t)aux % 16 == 0) && ((ldaux * esz) % 16 == 0);
  CUtensorMap tc = ta;
  if (store_mode && (rc = make_tmap(&tc, C, M, N, ldc, 32, c_dtype))) return rc;
  GemmArgs g;
  g.M = (int)M; g.N = (int)N; g.K = (int)K;
  g.C = C; g.ldc = ldc; g.bias = bias; g.epi = epi; g.aux = aux; g.ldaux = ldaux; g.accumulate = accumulate;
  g.kb_per_split = kb_per; g.splits = split_k;
  g.tiles_m = (int)ceil_div64(M, two ? 2 * BM : BM); g.tiles_n = (int)ceil_div64(N, BN);
  g.vec_ok = vec_ok; g.store_mode = store_mode;
  g.debug = e_dbg.geti("ICAP_GEMM_DEBUG", 0);
  g.b_static = b_static;
  g.trace = icap_trace_slot();
  if (epi == 3) return launch<256, false, true, true, bf16, true>(ta, tb, tc, g, st);   // the one row-statistics build
  auto go = [&](auto ak, auto bkm) {
    auto by_c = [&](auto bn, auto tw) {
      return dispatch_act(c_dtype, [&](auto tag) { return launch<bn, tw, ak, bkm, decltype(tag)>(ta, tb, tc, g, st); });
    };
    return two ? by_c(int_c<256>{}, std::true_type{})
               : BN == 256 ? by_c(int_c<256>{}, std::false_type{}) : by_c(int_c<128>{}, std::false_type{});
  };
  if (a_kmajor && b_kmajor) return go(std::true_type{}, std::true_type{});
  if (a_kmajor && !b_kmajor) return go(std::true_type{}, std::false_type{});
  return go(std::false_type{}, std::false_type{});
}
