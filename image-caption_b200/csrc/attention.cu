// Fused multi-head attention, forward and backward, one CTA per (batch, head).
//
//   S = (Q / sqrt(dk)) K^T ; masked_fill(-inf) ; P = softmax(S) ; P = dropout(P) ; O = P V
//
// Follows ScaledDotProductAttention.forward + the head split/merge of MultiHeadAttention.forward
// (modules.py:16-27, 72-84): q is scaled BEFORE QK^T, masks are True = masked, dropout is applied
// to the probabilities.  Masks are generated in-kernel: key j of batch b is masked iff
// kvalid[b*Lk+j] == 0 (kvalid may be null) or (causal and j > i)  (model.py:202-209,311-319,421-430).
// Heads are addressed in the packed projection outputs ([rows, H*dh] with a row stride), so no
// transpose / contiguous copies exist.  The whole (b, h) problem (L <= ~128) lives in shared memory;
// softmax uses warp shuffles.  Backward recomputes P (nothing but Q, K, V, dO is read).
#include <stdlib.h>
#include "icap_common.cuh"

namespace {

constexpr int NT = 128;

struct AttnDims {
  int Lq, Lk, LkP, dk, dv, H;
  int ldD;      // row stride of the dropout element index, attn_drop_ld(Lk) (the smem row stride is LkP)
};

template <typename T>
__device__ __forceinline__ void load_rows(float* dst, int dst_ld, const T* src, int64_t src_ld, int rows, int cols,
                                          float scale) {
  const int cq = cols >> 2;
  for (int u = threadIdx.x; u < rows * cq; u += NT) {
    const int r = u / cq, c = (u % cq) * 4;
    float v[4];
    load4(src + (int64_t)r * src_ld + c, v);
#pragma unroll
    for (int j = 0; j < 4; ++j) dst[r * dst_ld + c + j] = v[j] * scale;
  }
}
template <typename T>
__device__ __forceinline__ void load_rows_t(float* dst, int dst_ld, const T* src, int64_t src_ld, int rows, int cols) {
  // dst[c][r] = src[r][c]; columns beyond `rows` up to dst_ld are zeroed by the caller
  const int cq = cols >> 2;
  for (int u = threadIdx.x; u < rows * cq; u += NT) {
    const int r = u % rows, c = (u / rows) * 4;
    float v[4];
    load4(src + (int64_t)r * src_ld + c, v);
#pragma unroll
    for (int j = 0; j < 4; ++j) dst[(c + j) * dst_ld + r] = v[j];
  }
}

// P[i][j] for all i, j (softmax with masks, then dropout); P has row stride LkP, padded cols = 0
__device__ __forceinline__ void scores_softmax(float* P, float* Praw, const float* Qs, const float* Kt,
                                               const uint8_t* kvalid_b, const AttnDims& D, int causal, float p_drop,
                                               uint32_t thresh, uint64_t seed, uint64_t bh) {
  const int jq = D.LkP >> 2;
  for (int u = threadIdx.x; u < D.Lq * jq; u += NT) {
    const int i = u / jq, j0 = (u % jq) * 4;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    const float* q = Qs + i * D.dk;
    for (int c = 0; c < D.dk; ++c) {
      const float qc = q[c];
      const float4 k = *reinterpret_cast<const float4*>(Kt + c * D.LkP + j0);
      a0 = fmaf(qc, k.x, a0); a1 = fmaf(qc, k.y, a1); a2 = fmaf(qc, k.z, a2); a3 = fmaf(qc, k.w, a3);
    }
    *reinterpret_cast<float4*>(P + i * D.LkP + j0) = make_float4(a0, a1, a2, a3);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  for (int i = warp; i < D.Lq; i += NT / 32) {
    float* row = P + i * D.LkP;
    float mx = -INFINITY;
    for (int j = lane; j < D.LkP; j += 32) {
      const bool masked = (j >= D.Lk) || (kvalid_b && !kvalid_b[j]) || (causal && j > i);
      const float s = masked ? -INFINITY : row[j];
      row[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < D.LkP; j += 32) {
      const float e = (row[j] == -INFINITY) ? 0.f : expf(row[j] - mx);
      row[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;   // all-masked row -> inf/NaN exactly like the reference's softmax
    for (int j = lane; j < D.LkP; j += 32) {
      float p = row[j] * inv;
      if (j >= D.Lk) p = 0.f;
      if (Praw) Praw[i * D.LkP + j] = p;
      if (p_drop > 0.f) {
        const uint64_t e = (bh * D.Lq + i) * (uint64_t)D.ldD + j;
        const uint32_t keep = dropout_keep2(seed_fold(seed), e >> 1, thresh);
        p = ((keep >> (e & 1)) & 1u) ? p * keep_scale : 0.f;
      }
      row[j] = p;
    }
  }
  __syncthreads();
}

template <typename T>
__global__ void __launch_bounds__(NT)
mha_fwd_kernel(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, int64_t ldk, const T* __restrict__ v,
               int64_t ldv, T* __restrict__ o, int64_t ldo, const uint8_t* __restrict__ kvalid, AttnDims D, int causal,
               float p_drop, uint32_t thresh, uint64_t seed, const int* __restrict__ seed_dev,
               float* __restrict__ attn_mean) {
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x / D.H, h = blockIdx.x % D.H;
  float* Qs = sm;                         // [Lq][dk]
  float* Kt = Qs + D.Lq * D.dk;           // [dk][LkP]
  float* Vs = Kt + D.dk * D.LkP;          // [Lk][dv]
  float* P = Vs + D.Lk * D.dv;            // [Lq][LkP]
  for (int u = threadIdx.x; u < D.dk * D.LkP; u += NT) Kt[u] = 0.f;
  __syncthreads();
  load_rows(Qs, D.dk, q + (int64_t)b * D.Lq * ldq + h * D.dk, ldq, D.Lq, D.dk, (1.f / sqrtf((float)D.dk)));
  load_rows_t(Kt, D.LkP, k + (int64_t)b * D.Lk * ldk + h * D.dk, ldk, D.Lk, D.dk);
  load_rows(Vs, D.dv, v + (int64_t)b * D.Lk * ldv + h * D.dv, ldv, D.Lk, D.dv, 1.f);
  __syncthreads();
  scores_softmax(P, nullptr, Qs, Kt, kvalid ? kvalid + (int64_t)b * D.Lk : nullptr, D, causal, p_drop, thresh, seed,
                 (uint64_t)blockIdx.x);
  if (attn_mean) {   // mean over heads of the probabilities (greedy visualisation, model.py:123)
    for (int u = threadIdx.x; u < D.Lq * D.Lk; u += NT) {
      const int i = u / D.Lk, j = u % D.Lk;
      atomicAdd(attn_mean + ((int64_t)b * D.Lq + i) * D.Lk + j, P[i * D.LkP + j] / (float)D.H);
    }
  }
  const int cq = D.dv >> 2;
  for (int u = threadIdx.x; u < D.Lq * cq; u += NT) {
    const int i = u / cq, c0 = (u % cq) * 4;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const float* prow = P + i * D.LkP;
    for (int j = 0; j < D.Lk; ++j) {
      const float p = prow[j];
      const float4 vv = *reinterpret_cast<const float4*>(Vs + j * D.dv + c0);
      acc[0] = fmaf(p, vv.x, acc[0]); acc[1] = fmaf(p, vv.y, acc[1]);
      acc[2] = fmaf(p, vv.z, acc[2]); acc[3] = fmaf(p, vv.w, acc[3]);
    }
    store4(o + ((int64_t)b * D.Lq + i) * ldo + h * D.dv + c0, acc);
  }
}

template <typename T>
__global__ void __launch_bounds__(NT)
mha_bwd_kernel(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, int64_t ldk, const T* __restrict__ v,
               int64_t ldv, const T* __restrict__ dout, int64_t lddo, T* __restrict__ dq, int64_t lddq,
               T* __restrict__ dk_, int64_t lddk, T* __restrict__ dv_, int64_t lddv,
               const uint8_t* __restrict__ kvalid, AttnDims D, int causal, float p_drop, uint32_t thresh,
               uint64_t seed, const int* __restrict__ seed_dev) {
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x / D.H, h = blockIdx.x % D.H;
  float* Qs = sm;                          // [Lq][dk]  (pre-scaled)
  float* Kn = Qs + D.Lq * D.dk;            // [Lk][dk]
  float* Kt = Kn + D.Lk * D.dk;            // [dk][LkP]
  float* Vt = Kt + D.dk * D.LkP;           // [dv][LkP]
  float* dO = Vt + D.dv * D.LkP;           // [Lq][dv]
  float* Pd = dO + D.Lq * D.dv;            // [Lq][LkP]  dropped probabilities, later dS
  float* Pr = Pd + D.Lq * D.LkP;           // [Lq][LkP]  raw probabilities
  const float scale = (1.f / sqrtf((float)D.dk));
  for (int u = threadIdx.x; u < (D.dk + D.dv) * D.LkP; u += NT) Kt[u] = 0.f;   // Kt and Vt are adjacent
  __syncthreads();
  load_rows(Qs, D.dk, q + (int64_t)b * D.Lq * ldq + h * D.dk, ldq, D.Lq, D.dk, scale);
  load_rows(Kn, D.dk, k + (int64_t)b * D.Lk * ldk + h * D.dk, ldk, D.Lk, D.dk, 1.f);
  load_rows_t(Kt, D.LkP, k + (int64_t)b * D.Lk * ldk + h * D.dk, ldk, D.Lk, D.dk);
  load_rows_t(Vt, D.LkP, v + (int64_t)b * D.Lk * ldv + h * D.dv, ldv, D.Lk, D.dv);
  load_rows(dO, D.dv, dout + (int64_t)b * D.Lq * lddo + h * D.dv, lddo, D.Lq, D.dv, 1.f);
  __syncthreads();
  scores_softmax(Pd, Pr, Qs, Kt, kvalid ? kvalid + (int64_t)b * D.Lk : nullptr, D, causal, p_drop, thresh, seed,
                 (uint64_t)blockIdx.x);

  // dV[j][c] = sum_i Pd[i][j] dO[i][c]
  {
    const int cq = D.dv >> 2;
    for (int u = threadIdx.x; u < D.Lk * cq; u += NT) {
      const int j = u / cq, c0 = (u % cq) * 4;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int i = 0; i < D.Lq; ++i) {
        const float p = Pd[i * D.LkP + j];
        const float4 g = *reinterpret_cast<const float4*>(dO + i * D.dv + c0);
        acc[0] = fmaf(p, g.x, acc[0]); acc[1] = fmaf(p, g.y, acc[1]);
        acc[2] = fmaf(p, g.z, acc[2]); acc[3] = fmaf(p, g.w, acc[3]);
      }
      store4(dv_ + ((int64_t)b * D.Lk + j) * lddv + h * D.dv + c0, acc);
    }
  }
  __syncthreads();
  // dPd[i][j] = sum_c dO[i][c] V[j][c]; then dP = dropout-mask * dPd / (1-p), recovered from Pd/Pr
  {
    const int jq = D.LkP >> 2;
    for (int u = threadIdx.x; u < D.Lq * jq; u += NT) {
      const int i = u / jq, j0 = (u % jq) * 4;
      float a[4] = {0.f, 0.f, 0.f, 0.f};
      const float* g = dO + i * D.dv;
      for (int c = 0; c < D.dv; ++c) {
        const float gc = g[c];
        const float4 vv = *reinterpret_cast<const float4*>(Vt + c * D.LkP + j0);
        a[0] = fmaf(gc, vv.x, a[0]); a[1] = fmaf(gc, vv.y, a[1]);
        a[2] = fmaf(gc, vv.z, a[2]); a[3] = fmaf(gc, vv.w, a[3]);
      }
      // Pd = keep ? Pr/(1-p) : 0  =>  dP = keep ? dPd/(1-p) : 0 ;  P*dP = Pd * dPd
#pragma unroll
      for (int t = 0; t < 4; ++t) Pd[i * D.LkP + j0 + t] *= a[t];     // now holds P * dP
    }
  }
  __syncthreads();
  // dS[i][j] = P dP - P * sum_j (P dP)
  {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = warp; i < D.Lq; i += NT / 32) {
      float sum = 0.f;
      for (int j = lane; j < D.Lk; j += 32) sum += Pd[i * D.LkP + j];
      sum = warp_sum(sum);
      for (int j = lane; j < D.LkP; j += 32)
        Pd[i * D.LkP + j] = (j < D.Lk) ? Pd[i * D.LkP + j] - Pr[i * D.LkP + j] * sum : 0.f;
    }
  }
  __syncthreads();
  // dQ[i][c] = scale * sum_j dS[i][j] K[j][c]
  {
    const int cq = D.dk >> 2;
    for (int u = threadIdx.x; u < D.Lq * cq; u += NT) {
      const int i = u / cq, c0 = (u % cq) * 4;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int j = 0; j < D.Lk; ++j) {
        const float s = Pd[i * D.LkP + j];
        const float4 kk = *reinterpret_cast<const float4*>(Kn + j * D.dk + c0);
        acc[0] = fmaf(s, kk.x, acc[0]); acc[1] = fmaf(s, kk.y, acc[1]);
        acc[2] = fmaf(s, kk.z, acc[2]); acc[3] = fmaf(s, kk.w, acc[3]);
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) acc[t] *= scale;
      store4(dq + ((int64_t)b * D.Lq + i) * lddq + h * D.dk + c0, acc);
    }
    // dK[j][c] = sum_i dS[i][j] Qs[i][c]
    for (int u = threadIdx.x; u < D.Lk * cq; u += NT) {
      const int j = u / cq, c0 = (u % cq) * 4;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int i = 0; i < D.Lq; ++i) {
        const float s = Pd[i * D.LkP + j];
        const float4 qq = *reinterpret_cast<const float4*>(Qs + i * D.dk + c0);
        acc[0] = fmaf(s, qq.x, acc[0]); acc[1] = fmaf(s, qq.y, acc[1]);
        acc[2] = fmaf(s, qq.z, acc[2]); acc[3] = fmaf(s, qq.w, acc[3]);
      }
      store4(dk_ + ((int64_t)b * D.Lk + j) * lddk + h * D.dk + c0, acc);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// KV-cached decoding attention: one query per row, one warp per (row, head).
//   lanes own keys for the score / softmax phase, then own output columns for P.V
template <typename T>
__global__ void __launch_bounds__(NT)
mha_decode_kernel(int rows, int H, int Lk, int dk, int dv, const T* __restrict__ q, int64_t ldq,
                  const T* __restrict__ kc, int64_t ldk, const T* __restrict__ vc, int64_t ldv, int kv_rows_per_seq,
                  T* __restrict__ o, int64_t ldo, const int* __restrict__ slot, int64_t slot_ld,
                  const int* __restrict__ tokens, int64_t tok_ld, int pad_idx, const uint8_t* __restrict__ kvalid,
                  int rows_per_image, float* __restrict__ attn_mean) {
  pdl_prologue();
  extern __shared__ __align__(16) float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * (NT / 32) + warp;
  if (unit >= rows * H) return;
  const int row = unit / H, h = unit % H;
  float* qs = sm + warp * dk;
  const float scale = 1.f / sqrtf((float)dk);
  for (int c = lane; c < dk; c += 32) qs[c] = to_f32(q[(int64_t)row * ldq + h * dk + c]) * scale;
  __syncwarp();
  const bool self_mode = tokens != nullptr;             // self-attention over the KV cache
  const int seq = row / rows_per_image;                 // cross-attention: image index
  float p[4];
  float mx = -INFINITY;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const int j = jj * 32 + lane;
    float s = -INFINITY;
    if (j < Lk) {
      bool masked;
      int64_t krow;
      if (self_mode) {
        masked = tokens[(int64_t)row * tok_ld + j] == pad_idx;
        krow = (int64_t)(slot ? slot[(int64_t)row * slot_ld + j] : row) * kv_rows_per_seq + j;
      } else {
        masked = kvalid && !kvalid[(int64_t)seq * Lk + j];
        krow = (int64_t)seq * kv_rows_per_seq + j;
      }
      if (!masked) {
        const T* kp = kc + krow * ldk + h * dk;
        float acc = 0.f;
        for (int c = 0; c < dk; c += 4) {
          float kv4[4];
          load4(kp + c, kv4);
          acc = fmaf(qs[c], kv4[0], acc); acc = fmaf(qs[c + 1], kv4[1], acc);
          acc = fmaf(qs[c + 2], kv4[2], acc); acc = fmaf(qs[c + 3], kv4[3], acc);
        }
        s = acc;
      }
    }
    p[jj] = s;
    mx = fmaxf(mx, s);
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    p[jj] = (p[jj] == -INFINITY) ? 0.f : expf(p[jj] - mx);
    sum += p[jj];
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    p[jj] *= inv;
    const int j = jj * 32 + lane;
    if (attn_mean && j < Lk) atomicAdd(attn_mean + (int64_t)row * Lk + j, p[jj] / (float)H);
  }
  // P.V : every lane takes part in the probability broadcast (dv may be < 32), lanes own columns lane + 32*i
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int j = 0; j < Lk; ++j) {
    float pj = 0.f;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const float t = __shfl_sync(0xffffffffu, p[jj], j & 31);
      if ((j >> 5) == jj) pj = t;
    }
    if (pj == 0.f) continue;                      // warp-uniform
    int64_t vrow;
    if (self_mode) vrow = (int64_t)(slot ? slot[(int64_t)row * slot_ld + j] : row) * kv_rows_per_seq + j;
    else vrow = (int64_t)seq * kv_rows_per_seq + j;
    const T* vp = vc + vrow * ldv + h * dv;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c0 = lane + 32 * i;
      if (c0 < dv) acc[i] = fmaf(pj, to_f32(vp[c0]), acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c0 = lane + 32 * i;
    if (c0 < dv) o[(int64_t)row * ldo + h * dv + c0] = from_f32<T>(acc[i]);
  }
}


// ---------------------------------------------------------------------------------------------
// Fast KV-cached decoding attention for head dim 64 (dk == dv == 64), any dtype.
// One warp per (query group, head); a group = G queries that read the SAME keys/values:
//   cross-attention: the G = rows_per_image beams of one image (K/V of the image are read once, not per beam)
//   self-attention : G = 1 (every beam has its own cache rows through the slot table)
// K / V rows are 128 B (bf16) or 256 B (fp32): 8 lanes x 8 elements cover one row with 16-byte loads, so a warp
// reads 4 keys per load instruction, fully coalesced.  Scores are reduced over the 8 lanes of a key with three
// xor-shuffles, staged in shared memory for the softmax, then P.V accumulates 8 output columns per lane and is
// reduced over the 4 key sub-groups with two more shuffles.
constexpr int DEC_WARPS = 8, DEC_LK = 128;

template <typename T>
__device__ __forceinline__ void ld8(const T* p, float (&v)[8]);
template <>
__device__ __forceinline__ void ld8<float>(const float* p, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <>
__device__ __forceinline__ void ld8<bf16>(const bf16* p, float (&v)[8]) {
  const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
}
__device__ __forceinline__ void st8(float* p, const float (&v)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void st8(bf16* p, const float (&v)[8]) {
  uint4 t;
  __nv_bfloat162 h;
  h = __floats2bfloat162_rn(v[0], v[1]); t.x = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[2], v[3]); t.y = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[4], v[5]); t.z = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[6], v[7]); t.w = *reinterpret_cast<uint32_t*>(&h);
  *reinterpret_cast<uint4*>(p) = t;
}

template <typename T, int G>
__global__ void __launch_bounds__(DEC_WARPS * 32)
mha_decode64_kernel(int groups, int H, int Lk, const T* __restrict__ q, int64_t ldq, const T* __restrict__ kc,
                    int64_t ldk, const T* __restrict__ vc, int64_t ldv, int kv_rows_per_seq, T* __restrict__ o,
                    int64_t ldo, const int* __restrict__ slot, int64_t slot_ld, const int* __restrict__ tokens,
                    int64_t tok_ld, int pad_idx, const uint8_t* __restrict__ kvalid, float* __restrict__ attn_mean,
                    const T* __restrict__ knew, const T* __restrict__ vnew, int64_t ldn, int pos_new) {
  pdl_prologue();
  __shared__ float ps[DEC_WARPS][G][DEC_LK];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * DEC_WARPS + warp;
  if (unit >= groups * H) return;
  const int grp = unit / H, h = unit % H;
  const int sub = lane >> 3, ch = lane & 7;
  const bool self_mode = tokens != nullptr;      // G == 1: the group is the row
  float qv[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    ld8<T>(q + (int64_t)(grp * G + g) * ldq + h * 64 + ch * 8, qv[g]);
#pragma unroll
    for (int e = 0; e < 8; ++e) qv[g][e] *= 0.125f;                 // 1 / sqrt(64), applied to q as in modules.py:18
  }
  // ---- fused KV-cache append (self-attention): this row's new key / value of position pos_new go to its OWN cache
  // row (the slot table maps the newest position of a beam to the beam itself) and are used from registers below
  float knew_r[8], vnew_r[8];
  const bool append = knew != nullptr;
  if (append) {
    ld8<T>(knew + (int64_t)grp * ldn + h * 64 + ch * 8, knew_r);
    ld8<T>(vnew + (int64_t)grp * ldn + h * 64 + ch * 8, vnew_r);
    const int64_t crow = (int64_t)grp * kv_rows_per_seq + pos_new;
    if (sub == 0) st8(const_cast<T*>(kc) + crow * ldk + h * 64 + ch * 8, knew_r);
    if (sub == 1) st8(const_cast<T*>(vc) + crow * ldv + h * 64 + ch * 8, vnew_r);
  }
  // ---- physical cache row of every key (or -1 = masked), gathered up front: lane l owns keys l, l+32, ...
  // (tokens / slot / kvalid loads are coalesced and off the critical path of the K / V loads below)
  int kr[DEC_LK / 32];
#pragma unroll
  for (int jj = 0; jj < DEC_LK / 32; ++jj) {
    const int j = jj * 32 + lane;
    int r_ = -1;
    if (j < Lk) {
      if (self_mode) {
        const int sl = slot ? slot[(int64_t)grp * slot_ld + j] : grp;
        if (tokens[(int64_t)grp * tok_ld + j] != pad_idx) r_ = sl * kv_rows_per_seq + j;
      } else if (!(kvalid && !kvalid[(int64_t)grp * Lk + j])) {
        r_ = grp * kv_rows_per_seq + j;
      }
    }
    kr[jj] = r_;
  }
  constexpr int UB = 4;                              // key batches of 4 x 4: four independent 16-byte loads in flight
  // ---- scores
  for (int jb = 0; jb < Lk; jb += 4 * UB) {
    float kv[UB][8];
    int rr[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int j = jb + u * 4 + sub;                // < DEC_LK + 16: clamp the source lane, mask by j < Lk
      const int jj = (j >> 5) & (DEC_LK / 32 - 1);
      const int src = jj == 0 ? kr[0] : jj == 1 ? kr[1] : jj == 2 ? kr[2] : kr[3];
      const int got = __shfl_sync(0xffffffffu, src, j & 31);
      rr[u] = j < Lk ? got : -1;
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
#pragma unroll
      for (int e = 0; e < 8; ++e) kv[u][e] = 0.f;
      // branch-free: the four loads of a batch stay back to back; the appended position comes from registers
      const bool is_new = append && (jb + u * 4 + sub == pos_new);
      if (rr[u] >= 0 && !is_new) ld8<T>(kc + (int64_t)rr[u] * ldk + h * 64 + ch * 8, kv[u]);
#pragma unroll
      for (int e = 0; e < 8; ++e) kv[u][e] = (is_new && rr[u] >= 0) ? knew_r[e] : kv[u][e];
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int j = jb + u * 4 + sub;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float part = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) part = fmaf(qv[g][e], kv[u][e], part);
        part += __shfl_xor_sync(0xffffffffu, part, 1);
        part += __shfl_xor_sync(0xffffffffu, part, 2);
        part += __shfl_xor_sync(0xffffffffu, part, 4);
        if (ch == 0 && j < Lk) ps[warp][g][j] = rr[u] >= 0 ? part : -INFINITY;
      }
    }
  }
  __syncwarp();
  // ---- softmax over the keys, one query at a time (lanes own keys)
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float sv[DEC_LK / 32];
    float mx = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < DEC_LK / 32; ++jj) {
      const int j = jj * 32 + lane;
      sv[jj] = j < Lk ? ps[warp][g][j] : -INFINITY;
      mx = fmaxf(mx, sv[jj]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int jj = 0; jj < DEC_LK / 32; ++jj) {
      sv[jj] = (sv[jj] == -INFINITY) ? 0.f : expf(sv[jj] - mx);
      sum += sv[jj];
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
#pragma unroll
    for (int jj = 0; jj < DEC_LK / 32; ++jj) {
      const int j = jj * 32 + lane;
      if (j < Lk) {
        const float pj = sv[jj] * inv;
        ps[warp][g][j] = pj;
        if (attn_mean) atomicAdd(attn_mean + (int64_t)(grp * G + g) * Lk + j, pj / (float)H);
      }
    }
  }
  __syncwarp();
  // ---- P.V
  float acc[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[g][e] = 0.f;
  for (int jb = 0; jb < Lk; jb += 4 * UB) {
    float vv[UB][8];
    int rr[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int j = jb + u * 4 + sub;
      const int jj = (j >> 5) & (DEC_LK / 32 - 1);
      const int src = jj == 0 ? kr[0] : jj == 1 ? kr[1] : jj == 2 ? kr[2] : kr[3];
      const int got = __shfl_sync(0xffffffffu, src, j & 31);
      rr[u] = j < Lk ? got : -1;                     // masked keys have p == 0 for every query: never loaded
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
#pragma unroll
      for (int e = 0; e < 8; ++e) vv[u][e] = 0.f;
      const bool is_new = append && (jb + u * 4 + sub == pos_new);
      if (rr[u] >= 0 && !is_new) ld8<T>(vc + (int64_t)rr[u] * ldv + h * 64 + ch * 8, vv[u]);
#pragma unroll
      for (int e = 0; e < 8; ++e) vv[u][e] = (is_new && rr[u] >= 0) ? vnew_r[e] : vv[u][e];
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int j = jb + u * 4 + sub;
      if (rr[u] >= 0) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float pj = ps[warp][g][j];
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[g][e] = fmaf(pj, vv[u][e], acc[g][e]);
        }
      }
    }
  }
#pragma unroll
  for (int g = 0; g < G; ++g) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      acc[g][e] += __shfl_xor_sync(0xffffffffu, acc[g][e], 8);
      acc[g][e] += __shfl_xor_sync(0xffffffffu, acc[g][e], 16);
    }
    if (sub == 0) st8(o + (int64_t)(grp * G + g) * ldo + h * 64 + ch * 8, acc[g]);
  }
}


// ---------------------------------------------------------------------------------------------
// Self-attention decode step, "row per warp" mapping (head dim 64, width H*64 = WPR * 32 * EPL, at most 32 cached
// positions).  The warp-per-(row, head) kernel above spends ~700 instructions of fixed overhead per 64-wide head for
// <= 21 keys and was issue bound (ncu r1: 39 us per launch).  Here one warp owns EPL contiguous elements per lane of
// a row's K / V line (all or half of the heads at once): one fully coalesced 16/32-byte load per lane fetches a
// cached position for every head, the per-head dot product is reduced over the 64/EPL lanes of a head with xor
// shuffles, the softmax is online (running max / sum per head, kept redundantly in the head's lanes), and the new
// K / V of position pos_new are appended to the row's own cache line from registers.
template <typename T, int EPL> struct RawVec;                       // EPL elements as 16-byte words
template <int EPL> struct RawVec<bf16, EPL> { uint4 w[EPL / 8]; };
template <int EPL> struct RawVec<float, EPL> { uint4 w[EPL / 4]; };
template <typename T, int EPL>
__device__ __forceinline__ void raw_load(RawVec<T, EPL>& r, const T* p) {
#pragma unroll
  for (int i = 0; i < (int)(sizeof(r.w) / 16); ++i) r.w[i] = __ldg(reinterpret_cast<const uint4*>(p) + i);
}
template <typename T, int EPL>
__device__ __forceinline__ void raw_zero(RawVec<T, EPL>& r) {
#pragma unroll
  for (int i = 0; i < (int)(sizeof(r.w) / 16); ++i) r.w[i] = make_uint4(0u, 0u, 0u, 0u);
}
template <int EPL>
__device__ __forceinline__ void raw_unpack(const RawVec<bf16, EPL>& r, float (&v)[EPL]) {
#pragma unroll
  for (int i = 0; i < EPL / 8; ++i) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r.w[i]);
#pragma unroll
    for (int e = 0; e < 4; ++e) { v[i * 8 + 2 * e] = __low2float(h[e]); v[i * 8 + 2 * e + 1] = __high2float(h[e]); }
  }
}
template <int EPL>
__device__ __forceinline__ void raw_unpack(const RawVec<float, EPL>& r, float (&v)[EPL]) {
#pragma unroll
  for (int i = 0; i < EPL / 4; ++i) {
    v[i * 4] = __uint_as_float(r.w[i].x); v[i * 4 + 1] = __uint_as_float(r.w[i].y);
    v[i * 4 + 2] = __uint_as_float(r.w[i].z); v[i * 4 + 3] = __uint_as_float(r.w[i].w);
  }
}
template <int EPL>
__device__ __forceinline__ void raw_pack_store(bf16* p, const float (&v)[EPL]) {
#pragma unroll
  for (int i = 0; i < EPL / 8; ++i) {
    uint4 t;
    __nv_bfloat162 h;
    h = __floats2bfloat162_rn(v[i * 8 + 0], v[i * 8 + 1]); t.x = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(v[i * 8 + 2], v[i * 8 + 3]); t.y = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(v[i * 8 + 4], v[i * 8 + 5]); t.z = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(v[i * 8 + 6], v[i * 8 + 7]); t.w = *reinterpret_cast<uint32_t*>(&h);
    reinterpret_cast<uint4*>(p)[i] = t;
  }
}
template <int EPL>
__device__ __forceinline__ void raw_pack_store(float* p, const float (&v)[EPL]) {
#pragma unroll
  for (int i = 0; i < EPL / 4; ++i) reinterpret_cast<float4*>(p)[i] = make_float4(v[i * 4], v[i * 4 + 1], v[i * 4 + 2], v[i * 4 + 3]);
}


template <typename T, int EPL, int ROW_UB>      // ROW_UB: cached positions fetched per batch (loads in flight per lane)
__global__ void __launch_bounds__(320, 2)
mha_decode_row_kernel(int rows, int wpr, int Lk, const T* __restrict__ q, int64_t ldq, T* __restrict__ kc, int64_t ldk,
                      T* __restrict__ vc, int64_t ldv, int kv_rows_per_seq, T* __restrict__ o, int64_t ldo,
                      const int* __restrict__ slot, int64_t slot_ld, const int* __restrict__ tokens, int64_t tok_ld,
                      int pad_idx, const T* __restrict__ knew, const T* __restrict__ vnew, int64_t ldn, int pos_new) {
  constexpr int LPH = 64 / EPL;                       // lanes per head
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int row = gw / wpr, part = gw % wpr;          // part: which 32*EPL-wide slice of the row this warp owns
  const bool live = row < rows;
  const int col = (part * 32 + lane) * EPL;           // first element of this lane within a K / V / q / o row
  // lane l: physical cache row of position l, or -1 (position masked / beyond Lk).  The cached positions 0..pos_new-1
  // are pulled into L2 BEFORE the grid dependency resolves, i.e. while the QKV projection of this step is still running
  // on the tensor cores (its HBM traffic is small, this kernel's is all there is).  The token buffer and the slot table
  // that locate them may still be in flight at that point: in beam search the kernel that starts the step
  // (icap_decode_embed_ln) writes them, and the QKV GEMM in between lets this kernel become resident before it waits.
  // So the pre-wait lookup only steers the prefetch (a stale row costs bandwidth, never a wrong result) and the lookup
  // is repeated after griddepcontrol.wait for the loads that feed the result.  Both read through L2 (ld.global.cg):
  // the early read must not leave a stale line in L1 for the second one to hit.
  auto cache_row = [&]() {
    int r = -1;
    if (live && lane < Lk) {                          // both loads in flight together
      const int tk = __ldcg(tokens + (int64_t)row * tok_ld + lane);
      const int sl = slot ? __ldcg(slot + (int64_t)row * slot_ld + lane) : row;
      if (tk != pad_idx) r = sl * kv_rows_per_seq + lane;
    }
    return r;
  };
  int myrow = cache_row();
  for (int j = 0; j < Lk; ++j) {
    const int r = __shfl_sync(0xffffffffu, myrow, j);
    if (r >= 0 && j != pos_new) {
      asm volatile("prefetch.global.L2 [%0];" ::"l"(kc + (int64_t)r * ldk + col));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(vc + (int64_t)r * ldv + col));
    }
  }
  pdl_prologue();
  if (!live) return;
  myrow = cache_row();                                // tokens / slot of this step are final now
  float qv[EPL];
  {
    RawVec<T, EPL> r;
    raw_load<T, EPL>(r, q + (int64_t)row * ldq + col);
    raw_unpack(r, qv);
#pragma unroll
    for (int e = 0; e < EPL; ++e) qv[e] *= 0.125f;    // 1 / sqrt(64) on q, as modules.py:18
  }
  RawVec<T, EPL> knew_r, vnew_r;
  raw_load<T, EPL>(knew_r, knew + (int64_t)row * ldn + col);
  raw_load<T, EPL>(vnew_r, vnew + (int64_t)row * ldn + col);
  {
    const int64_t crow = (int64_t)row * kv_rows_per_seq + pos_new;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(knew_r.w) / 16); ++i) {
      reinterpret_cast<uint4*>(kc + crow * ldk + col)[i] = knew_r.w[i];
      reinterpret_cast<uint4*>(vc + crow * ldv + col)[i] = vnew_r.w[i];
    }
  }
  // ---- one pass over the cached positions, ROW_UB at a time: K and V of a batch are fetched together (2 * ROW_UB
  // independent loads in flight per lane), scores go through an online softmax (running max m / sum l, rescaled
  // accumulator), so there is a single memory round trip per batch instead of one for Q.K^T and one for P.V
  float acc[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) acc[e] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;
#pragma unroll
  for (int jb = 0; jb < 32; jb += ROW_UB) {
    if (jb < Lk) {                                    // warp-uniform
      RawVec<T, EPL> kraw[ROW_UB], vraw[ROW_UB];
      int rr[ROW_UB];
#pragma unroll
      for (int u = 0; u < ROW_UB; ++u) {
        rr[u] = __shfl_sync(0xffffffffu, myrow, jb + u);
        raw_zero<T, EPL>(kraw[u]);
        raw_zero<T, EPL>(vraw[u]);
        if (rr[u] >= 0 && jb + u != pos_new) {
          raw_load<T, EPL>(kraw[u], kc + (int64_t)rr[u] * ldk + col);
          raw_load<T, EPL>(vraw[u], vc + (int64_t)rr[u] * ldv + col);
        }
      }
      float sb[ROW_UB];
      float bmax = -INFINITY;
#pragma unroll
      for (int u = 0; u < ROW_UB; ++u) {
        sb[u] = -INFINITY;
        if (jb + u < Lk) {                            // warp-uniform
          float kv[EPL];
          if (jb + u == pos_new) raw_unpack(knew_r, kv); else raw_unpack(kraw[u], kv);
          float part_s = 0.f;
#pragma unroll
          for (int e = 0; e < EPL; ++e) part_s = fmaf(qv[e], kv[e], part_s);
#pragma unroll
          for (int off = 1; off < LPH; off <<= 1) part_s += __shfl_xor_sync(0xffffffffu, part_s, off);
          if (rr[u] >= 0) sb[u] = part_s;
          bmax = fmaxf(bmax, sb[u]);
        }
      }
      const float m_new = fmaxf(m_run, bmax);
      if (m_new != -INFINITY) {                       // identical in the lanes of a head; other heads may differ
        const float rescale = (m_run == -INFINITY) ? 0.f : __expf(m_run - m_new);
        l_run *= rescale;
#pragma unroll
        for (int e = 0; e < EPL; ++e) acc[e] *= rescale;
#pragma unroll
        for (int u = 0; u < ROW_UB; ++u) {
          if (jb + u < Lk) {
            const float pj = (sb[u] == -INFINITY) ? 0.f : __expf(sb[u] - m_new);
            l_run += pj;
            float vv[EPL];
            if (jb + u == pos_new) raw_unpack(vnew_r, vv); else raw_unpack(vraw[u], vv);
#pragma unroll
            for (int e = 0; e < EPL; ++e) acc[e] = fmaf(pj, vv[e], acc[e]);
          }
        }
        m_run = m_new;
      }
    }
  }
  {
    const float inv = 1.f / l_run;                    // all keys masked -> inf/NaN exactly like the reference's softmax
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc[e] *= inv;
  }
  raw_pack_store<EPL>(o + (int64_t)row * ldo + col, acc);
}

// ---------------------------------------------------------------------------------------------
// Cross-attention of a decode step, ONE CTA PER IMAGE (bf16, head dim 64, K | V rows contiguous as the packed
// projection [B*R, dk_tot + dv_tot] leaves them): the G beam rows of an image attend the image's Lk region keys.
//   * the image's K|V block is ONE contiguous range of global memory: a single `cp.async.bulk` (TMA, 1-D) per chunk of
//     rows brings it into shared memory -- 72 KB in flight per CTA, two or three CTAs per SM, instead of 4096 tiny
//     (image, head) blocks with a few dependent 16-byte loads each (r2 timeline: 24 us per launch, 14 us exposed);
//   * only rows up to the last valid region are fetched (padded regions are a suffix in the reference's data);
//   * K/V of the regions are produced once per decode, long before this launch, so the first chunk is requested BEFORE
//     `griddepcontrol.wait`: it streams in while the kernel that produces q is still running;
//   * warp h owns head h: lane = (key slot 0..3, 16-byte chunk 0..7); every key slot keeps its own online-softmax state
//     (m, l, acc) over the keys j = slot (mod 4); the four states are merged once at the end (flash-decoding merge).
// Replaces ScaledDotProductAttention for the decoder->region attention inside the decode loops (modules.py:16-27,196-200).
constexpr int XI_MAXK = 128;            // keys per image
constexpr int XI_SMEM_MAX = 96 * 1024;  // K|V rows staged per chunk

__device__ __forceinline__ void xi_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  } while (!done);
}

template <int G>
__global__ void __launch_bounds__(512)
mha_cross_img_kernel(int H, int Lk, const bf16* __restrict__ q, int64_t ldq, const bf16* __restrict__ kv, int64_t ldkv,
                     int dk_tot, bf16* __restrict__ o, int64_t ldo, const uint8_t* __restrict__ kvalid, int chunk_rows) {
  extern __shared__ __align__(128) uint8_t xi_smem[];
  __shared__ __align__(8) unsigned long long xi_bar;
  __shared__ uint8_t s_valid[XI_MAXK];
  __shared__ int s_nlast;
  const int img = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&xi_bar);
  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(xi_smem);
  const int row_bytes = (int)ldkv * 2;
  // kvalid is written once per decode (encoder prologue), like K/V: safe to read before the grid dependency resolves
  if (threadIdx.x < XI_MAXK) s_valid[threadIdx.x] = (threadIdx.x < Lk && (!kvalid || kvalid[(int64_t)img * Lk + threadIdx.x])) ? 1 : 0;
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == 0) {
    int last = 0;
    for (int j = lane; j < Lk; j += 32) if (s_valid[j]) last = j + 1;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, off));
    if (lane == 0) {
      s_nlast = last;
      const int rows0 = min(last, chunk_rows);
      if (rows0 > 0) {
        const uint32_t bytes = (uint32_t)(rows0 * row_bytes);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(sbase), "l"(kv + (int64_t)img * Lk * ldkv), "r"(bytes), "r"(bar) : "memory");
      }
    }
  }
  pdl_prologue();                       // q (and the buffer o is recycled from) depends on the preceding kernels
  __syncthreads();
  const int nlast = s_nlast;
  const int sub = lane >> 3, ch = lane & 7;
  float qv[G][8], acc[G][8], m_run[G], l_run[G];
  if (warp < H) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const uint4 t = __ldg(reinterpret_cast<const uint4*>(q + (int64_t)(img * G + g) * ldq + warp * 64 + ch * 8));
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        qv[g][2 * i] = __low2float(h2[i]) * 0.125f;           // 1 / sqrt(64) on q, as modules.py:18
        qv[g][2 * i + 1] = __high2float(h2[i]) * 0.125f;
      }
      m_run[g] = -INFINITY; l_run[g] = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[g][e] = 0.f;
    }
  }
  int chunk = 0;
  for (int j0 = 0; j0 < nlast; j0 += chunk_rows, ++chunk) {
    const int cr = min(chunk_rows, nlast - j0);
    if (chunk > 0) {
      __syncthreads();                  // every warp is done with the previous chunk
      if (threadIdx.x == 0) {
        const uint32_t bytes = (uint32_t)(cr * row_bytes);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(sbase), "l"(kv + ((int64_t)img * Lk + j0) * ldkv), "r"(bytes), "r"(bar) : "memory");
      }
    }
    xi_mbar_wait(bar, (uint32_t)(chunk & 1));
    if (warp < H) {
      for (int i = 0; i < cr; i += 4) {
        const int jl = i + sub, j = j0 + jl;
        const bool valid = jl < cr && s_valid[j];
        // every lane runs the same instruction stream (full-mask shuffles): an idle key slot multiplies zeros and
        // leaves its state alone
        uint4 kr = make_uint4(0u, 0u, 0u, 0u), vr = make_uint4(0u, 0u, 0u, 0u);
        if (valid) {
          const uint32_t ka = sbase + (uint32_t)(jl * row_bytes + (warp * 64 + ch * 8) * 2);
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(kr.x), "=r"(kr.y), "=r"(kr.z), "=r"(kr.w) : "r"(ka));
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(vr.x), "=r"(vr.y), "=r"(vr.z), "=r"(vr.w)
                       : "r"(ka + (uint32_t)dk_tot * 2u));
        }
        float kf[8], vf[8];
        const __nv_bfloat162* k2 = reinterpret_cast<const __nv_bfloat162*>(&kr);
        const __nv_bfloat162* v2 = reinterpret_cast<const __nv_bfloat162*>(&vr);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          kf[2 * t] = __low2float(k2[t]); kf[2 * t + 1] = __high2float(k2[t]);
          vf[2 * t] = __low2float(v2[t]); vf[2 * t + 1] = __high2float(v2[t]);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float sc = 0.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) sc = fmaf(qv[g][e], kf[e], sc);
          sc += __shfl_xor_sync(0xffffffffu, sc, 1);          // over the 8 lanes of this key slot
          sc += __shfl_xor_sync(0xffffffffu, sc, 2);
          sc += __shfl_xor_sync(0xffffffffu, sc, 4);
          if (valid) {
            const float m_new = fmaxf(m_run[g], sc);
            const float scale = __expf(m_run[g] - m_new), pj = __expf(sc - m_new);     // exp(-inf) = 0 on the first key
            l_run[g] = l_run[g] * scale + pj;
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[g][e] = fmaf(pj, vf[e], acc[g][e] * scale);
            m_run[g] = m_new;
          }
        }
      }
    }
  }
  if (warp < H) {
    // merge the four key-slot states (lanes l, l^8, l^16, l^24 hold the same dims of the same head)
    __syncwarp();
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
      for (int off = 8; off <= 16; off <<= 1) {
        const float mo = __shfl_xor_sync(0xffffffffu, m_run[g], off), lo = __shfl_xor_sync(0xffffffffu, l_run[g], off);
        const float m_new = fmaxf(m_run[g], mo);
        const float sa = (m_run[g] == -INFINITY) ? 0.f : __expf(m_run[g] - m_new);
        const float sb = (mo == -INFINITY) ? 0.f : __expf(mo - m_new);
        l_run[g] = l_run[g] * sa + lo * sb;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float ao = __shfl_xor_sync(0xffffffffu, acc[g][e], off);
          acc[g][e] = acc[g][e] * sa + ao * sb;
        }
        m_run[g] = m_new;
      }
      if (sub == 0) {
        const float inv = 1.f / l_run[g];             // all keys masked -> inf/NaN exactly like the reference's softmax
        float ov[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) ov[e] = acc[g][e] * inv;
        st8(o + (int64_t)(img * G + g) * ldo + warp * 64 + ch * 8, ov);
      }
    }
  }
}

template <int G>
int launch_cross_img(int64_t images, int64_t H, int64_t Lk, const void* q, int64_t ldq, const void* kv, int64_t ldkv,
                     int64_t dk_tot, void* o, int64_t ldo, const uint8_t* kvalid, cudaStream_t st) {
  const int row_bytes = (int)ldkv * 2;
  int chunk_rows = XI_SMEM_MAX / row_bytes;
  if (chunk_rows > Lk) chunk_rows = (int)Lk;
  const size_t smem = (size_t)chunk_rows * row_bytes;
  if (int rc = ensure_smem<mha_cross_img_kernel<G>>(smem)) return rc;
  icap_launch(mha_cross_img_kernel<G>, (unsigned)images, (unsigned)(32 * H), smem, st, H, Lk, q, ldq, kv, ldkv, dk_tot, o, ldo,
              kvalid, chunk_rows);
  ICAP_LAUNCH_CHECK("icap_mha_decode(cross, image per CTA)");
  return 0;
}

template <typename T, int G>
int launch_decode64(int64_t groups, int64_t H, int64_t Lk, const void* q, int64_t ldq, const void* kc, int64_t ldk,
                    const void* vc, int64_t ldv, int64_t kv_rows_per_seq, void* o, int64_t ldo, const int* slot,
                    int64_t slot_ld, const int* tokens, int64_t tok_ld, int pad_idx, const uint8_t* kvalid,
                    float* attn_mean, cudaStream_t st, const void* knew = nullptr, const void* vnew = nullptr,
                    int64_t ldn = 0, int pos_new = 0) {
  const unsigned grid = (unsigned)ceil_div64(groups * H, DEC_WARPS);
  icap_launch(mha_decode64_kernel<T, G>, grid, DEC_WARPS * 32, 0, st, groups, H, Lk, q, ldq, kc, ldk, vc, ldv, kv_rows_per_seq,
              o, ldo, slot, slot_ld, tokens, tok_ld, pad_idx, kvalid, attn_mean, knew, vnew, ldn, pos_new);
  ICAP_LAUNCH_CHECK("icap_mha_decode(64)");
  return 0;
}

int check_dims(const char* fn, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv) {
  ICAP_ARG(B > 0 && H > 0 && Lq > 0 && Lk > 0, "%s: empty problem", fn);
  ICAP_ARG(dk % 4 == 0 && dv % 4 == 0 && dk > 0 && dv > 0, "%s: head dims must be multiples of 4 (dk=%lld dv=%lld)", fn,
           (long long)dk, (long long)dv);
  return 0;
}

}  // namespace

extern "C" int icap_mha_fwd(int dtype, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv,
                            const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            void* o, int64_t ldo, const uint8_t* kvalid, int causal, float p_drop, uint64_t seed,
                            const int* seed_dev, float* attn_mean, void* stream) {
  if (int rc = check_dims("icap_mha_fwd", B, H, Lq, Lk, dk, dv)) return rc;
  if (attn_mean == nullptr && icap_mha_mma_ok(dtype, Lq, Lk, dk, dv, ldq, ldk, ldv, q, k, v) && ldo % 8 == 0 &&
      (uintptr_t)o % 16 == 0)
    return icap_mha_fwd_mma(B, H, Lq, Lk, q, ldq, k, ldk, v, ldv, o, ldo, kvalid, causal, p_drop, seed, seed_dev,
                            (cudaStream_t)stream);
  AttnDims D{(int)Lq, (int)Lk, (int)((Lk + 3) & ~3), (int)dk, (int)dv, (int)H, attn_drop_ld(Lk)};
  const size_t smem = sizeof(float) * ((size_t)D.Lq * D.dk + (size_t)D.dk * D.LkP + (size_t)D.Lk * D.dv +
                                       (size_t)D.Lq * D.LkP);
  ICAP_ARG(smem <= 227 * 1024, "icap_mha_fwd: (Lq=%d, Lk=%d, dk=%d, dv=%d) needs %zu B of shared memory", D.Lq, D.Lk,
           D.dk, D.dv, smem);
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t th = dropout_threshold(p_drop);
  const int rc = dispatch_act(dtype, [&](auto tag) {
    if (int rc = ensure_smem<mha_fwd_kernel<decltype(tag)>>(smem)) return rc;
    icap_launch(mha_fwd_kernel<decltype(tag)>, (unsigned)(B * H), NT, smem, st, q, ldq, k, ldk, v, ldv, o, ldo, kvalid, D, causal,
                p_drop, th, seed, seed_dev, attn_mean);
    return 0;
  });
  if (rc) return rc;
  ICAP_LAUNCH_CHECK("icap_mha_fwd");
  return 0;
}

extern "C" int icap_mha_bwd(int dtype, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv,
                            const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            const void* dout, int64_t lddo, void* dq, int64_t lddq, void* dk_out, int64_t lddk,
                            void* dv_out, int64_t lddv, const uint8_t* kvalid, int causal, float p_drop, uint64_t seed,
                            const int* seed_dev, void* stream) {
  if (int rc = check_dims("icap_mha_bwd", B, H, Lq, Lk, dk, dv)) return rc;
  if (icap_mha_mma_ok(dtype, Lq, Lk, dk, dv, ldq, ldk, ldv, q, k, v) && lddo % 8 == 0 && lddq % 8 == 0 &&
      lddk % 8 == 0 && lddv % 8 == 0 && (uintptr_t)dout % 16 == 0 && (uintptr_t)dq % 16 == 0 &&
      (uintptr_t)dk_out % 16 == 0 && (uintptr_t)dv_out % 16 == 0)
    return icap_mha_bwd_mma(B, H, Lq, Lk, q, ldq, k, ldk, v, ldv, dout, lddo, dq, lddq, dk_out, lddk, dv_out, lddv,
                            kvalid, causal, p_drop, seed, seed_dev, (cudaStream_t)stream);
  AttnDims D{(int)Lq, (int)Lk, (int)((Lk + 3) & ~3), (int)dk, (int)dv, (int)H, attn_drop_ld(Lk)};
  const size_t smem = sizeof(float) * ((size_t)D.Lq * D.dk + (size_t)D.Lk * D.dk + (size_t)D.dk * D.LkP +
                                       (size_t)D.dv * D.LkP + (size_t)D.Lq * D.dv + 2 * (size_t)D.Lq * D.LkP);
  ICAP_ARG(smem <= 227 * 1024, "icap_mha_bwd: (Lq=%d, Lk=%d, dk=%d, dv=%d) needs %zu B of shared memory", D.Lq, D.Lk,
           D.dk, D.dv, smem);
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t th = dropout_threshold(p_drop);
  const int rc = dispatch_act(dtype, [&](auto tag) {
    if (int rc = ensure_smem<mha_bwd_kernel<decltype(tag)>>(smem)) return rc;
    icap_launch(mha_bwd_kernel<decltype(tag)>, (unsigned)(B * H), NT, smem, st, q, ldq, k, ldk, v, ldv, dout, lddo, dq, lddq,
                dk_out, lddk, dv_out, lddv, kvalid, D, causal, p_drop, th, seed, seed_dev);
    return 0;
  });
  if (rc) return rc;
  ICAP_LAUNCH_CHECK("icap_mha_bwd");
  return 0;
}

extern "C" int icap_mha_decode(int dtype, int64_t rows, int64_t H, int64_t Lk, int64_t dk, int64_t dv, const void* q,
                               int64_t ldq, const void* kc, int64_t ldk, const void* vc, int64_t ldv,
                               int64_t kv_rows_per_seq, void* o, int64_t ldo, const int* slot, int64_t slot_ld,
                               const int* tokens, int64_t tok_ld, int pad_idx, const uint8_t* kvalid,
                               int64_t rows_per_image, float* attn_mean, void* stream) {
  if (int rc = check_dims("icap_mha_decode", rows, H, 1, Lk, dk, dv)) return rc;
  ICAP_ARG(Lk <= 128, "icap_mha_decode: at most 128 keys per query (got %lld)", (long long)Lk);
  ICAP_ARG(dv <= 128, "icap_mha_decode: head dim of V must be <= 128 (got %lld)", (long long)dv);
  ICAP_ARG(slot == nullptr || tokens != nullptr, "icap_mha_decode: a slot table needs the token buffer (self mode)");
  ICAP_ARG(rows_per_image >= 1, "icap_mha_decode: rows_per_image must be >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int esz = dtype == ICAP_F32 ? 4 : 2;
  const bool al = ((uintptr_t)q % 16 == 0) && ((uintptr_t)kc % 16 == 0) && ((uintptr_t)vc % 16 == 0) &&
                  ((uintptr_t)o % 16 == 0) && (ldq * esz) % 16 == 0 && (ldk * esz) % 16 == 0 && (ldv * esz) % 16 == 0 &&
                  (ldo * esz) % 16 == 0;
  // cross-attention, K | V rows contiguous (the packed projection), head dim 64: one CTA per image, TMA bulk staging
  if (tokens == nullptr && attn_mean == nullptr && dtype == ICAP_BF16 && dk == 64 && dv == 64 && al && H <= 16 &&
      Lk <= XI_MAXK && kv_rows_per_seq == Lk && rows % rows_per_image == 0 && ldk == ldv &&
      (const bf16*)vc == (const bf16*)kc + H * dk && ldk * 2 <= XI_SMEM_MAX && (ldk * 2) % 16 == 0 &&
      (rows_per_image <= 5 || rows_per_image == 8) && env_flag<7>("ICAP_DECODE_IMG_CROSS")) {
    const int64_t images = rows / rows_per_image;
    auto go = [&](auto g) { return launch_cross_img<g>(images, H, Lk, q, ldq, kc, ldk, H * dk, o, ldo, kvalid, st); };
    switch (rows_per_image) {
      case 1: return go(int_c<1>{});
      case 2: return go(int_c<2>{});
      case 3: return go(int_c<3>{});
      case 4: return go(int_c<4>{});
      case 5: return go(int_c<5>{});
      default: return go(int_c<8>{});
    }
  }
  // cross-attention of a beam group = a tiny full attention (Lq = beams, Lk = regions, shared K/V): tensor-core
  // kernel (mma.sync), ~5x fewer instructions than the SIMT path for 5 beams x 36 regions x 64 dims
  if (tokens == nullptr && attn_mean == nullptr && rows_per_image >= 2 && rows % rows_per_image == 0 &&
      kv_rows_per_seq == Lk && ldo % 8 == 0 && (uintptr_t)o % 16 == 0 &&
      icap_mha_mma_ok(dtype, rows_per_image, Lk, dk, dv, ldq, ldk, ldv, q, kc, vc) && !env_flag<0>("ICAP_DECODE_NO_MMA"))
    return icap_mha_fwd_mma(rows / rows_per_image, H, rows_per_image, Lk, q, ldq, kc, ldk, vc, ldv, o, ldo, kvalid, 0, 0.f,
                            0, nullptr, st, /*kv_static=*/1);
  if (dk == 64 && dv == 64 && al && !env_flag<1>("ICAP_DECODE_SLOW")) {
    // group size: beams of one image share K/V in cross-attention; self-attention rows are independent
    int64_t G = tokens ? 1 : rows_per_image;
    if (G > 8 || rows % G != 0 || (G > 5 && G != 8)) G = 1;
    const int64_t groups = rows / G;
    // odd beam sizes (6, 7, > 8) in cross mode fall through to the generic kernel below
    if (tokens != nullptr || G == rows_per_image) {
      auto go = [&](auto g) {
        return dispatch_act(dtype, [&](auto tag) {
          return launch_decode64<decltype(tag), g>(groups, H, Lk, q, ldq, kc, ldk, vc, ldv, kv_rows_per_seq, o, ldo, slot,
                                                   slot_ld, tokens, tok_ld, pad_idx, kvalid, attn_mean, st);
        });
      };
      switch (G) {
        case 1: return go(int_c<1>{});
        case 2: return go(int_c<2>{});
        case 3: return go(int_c<3>{});
        case 4: return go(int_c<4>{});
        case 5: return go(int_c<5>{});
        case 8: return go(int_c<8>{});
        default: break;
      }
    }
  }
  const size_t smem = (NT / 32) * dk * sizeof(float);
  const unsigned grid = (unsigned)ceil_div64(rows * H, NT / 32);
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(mha_decode_kernel<decltype(tag)>, grid, NT, smem, st, rows, H, Lk, dk, dv, q, ldq, kc, ldk, vc, ldv,
                kv_rows_per_seq, o, ldo, slot, slot_ld, tokens, tok_ld, pad_idx, kvalid, rows_per_image, attn_mean);
  });
  ICAP_LAUNCH_CHECK("icap_mha_decode");
  return 0;
}

// Self-attention decode step with the KV-cache append fused in: K/V of position `pos` (k_new / v_new rows, leading
// dimension ld_new) are written to the row's own cache line and attended together with positions 0..pos-1.
extern "C" int icap_mha_decode_self(int dtype, int64_t rows, int64_t H, int64_t pos, int64_t dk, int64_t dv, const void* q,
                                    int64_t ldq, const void* k_new, const void* v_new, int64_t ld_new, void* kc,
                                    int64_t ldk, void* vc, int64_t ldv, int64_t kv_rows_per_seq, void* o, int64_t ldo,
                                    const int* slot, int64_t slot_ld, const int* tokens, int64_t tok_ld, int pad_idx,
                                    int64_t rows_per_image, void* stream) {
  if (int rc = check_dims("icap_mha_decode_self", rows, H, 1, pos + 1, dk, dv)) return rc;
  ICAP_ARG(pos >= 0 && pos < kv_rows_per_seq && pos + 1 <= 128, "icap_mha_decode_self: position %lld out of range", (long long)pos);
  ICAP_ARG(tokens && k_new && v_new && kc && vc, "icap_mha_decode_self: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int esz = dtype == ICAP_F32 ? 4 : 2;
  const bool al = ((uintptr_t)q % 16 == 0) && ((uintptr_t)kc % 16 == 0) && ((uintptr_t)vc % 16 == 0) &&
                  ((uintptr_t)o % 16 == 0) && ((uintptr_t)k_new % 16 == 0) && ((uintptr_t)v_new % 16 == 0) &&
                  (ldq * esz) % 16 == 0 && (ldk * esz) % 16 == 0 && (ldv * esz) % 16 == 0 && (ldo * esz) % 16 == 0 &&
                  (ld_new * esz) % 16 == 0;
  if (dk == 64 && dv == 64 && al && pos + 1 <= 32 && (H * 64) % 256 == 0 && !env_flag<1>("ICAP_DECODE_SLOW") &&
      !env_flag<2>("ICAP_DECODE_NO_ROW")) {
    // row-per-warp kernel: EPL elements per lane, wpr warps per row
    static IcapEnv e_ub;
    const int ub_env = e_ub.geti("ICAP_DECODE_UB", 4);
    const int width = (int)(H * 64);
    constexpr int epl = 8;
    const int wpr = width / (32 * epl);
    // Block = the rows of whole images (beams of an image share most of their prefix through the slot table: the same
    // physical cache lines are then fetched by warps of ONE block at about the same time and hit in L1); 8 warps
    // otherwise.  The kernel derives (row, part) from the global warp number, so any block size works.
    int wpb = 8;
    if (rows_per_image > 1 && rows % rows_per_image == 0 && rows_per_image * wpr <= 10 && !env_flag<5>("ICAP_DECODE_NO_IMG_BLOCKS"))
      wpb = (int)rows_per_image * wpr;
    const unsigned grid = (unsigned)ceil_div64(rows * wpr, wpb);
    const unsigned nthr = (unsigned)(32 * wpb);
    dispatch_act(dtype, [&](auto tag) {
      auto go = [&](auto ub) {
        icap_launch(mha_decode_row_kernel<decltype(tag), 8, ub>, grid, nthr, 0, st, rows, wpr, pos + 1, q, ldq, kc, ldk, vc, ldv,
                    kv_rows_per_seq, o, ldo, slot, slot_ld, tokens, tok_ld, pad_idx, k_new, v_new, ld_new, pos);
      };
      if (ub_env == 8) go(int_c<8>{}); else go(int_c<4>{});
    });
    ICAP_LAUNCH_CHECK("icap_mha_decode_self(row)");
    return 0;
  }
  if (dk == 64 && dv == 64 && al && !env_flag<1>("ICAP_DECODE_SLOW")) {
    return dispatch_act(dtype, [&](auto tag) {
      return launch_decode64<decltype(tag), 1>(rows, H, pos + 1, q, ldq, kc, ldk, vc, ldv, kv_rows_per_seq, o, ldo, slot,
                                               slot_ld, tokens, tok_ld, pad_idx, nullptr, nullptr, st, k_new, v_new, ld_new,
                                               (int)pos);
    });
  }
  // generic path: strided copies into the cache, then the plain decode attention
  if (int rc = icap_copy2d(k_new, dtype, ld_new, (char*)kc + pos * ldk * esz, dtype, kv_rows_per_seq * ldk, rows, H * dk, 0, stream))
    return rc;
  if (int rc = icap_copy2d(v_new, dtype, ld_new, (char*)vc + pos * ldv * esz, dtype, kv_rows_per_seq * ldv, rows, H * dv, 0, stream))
    return rc;
  return icap_mha_decode(dtype, rows, H, pos + 1, dk, dv, q, ldq, kc, ldk, vc, ldv, kv_rows_per_seq, o, ldo, slot, slot_ld,
                         tokens, tok_ld, pad_idx, nullptr, 1, nullptr, stream);
}
