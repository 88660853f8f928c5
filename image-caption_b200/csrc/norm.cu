// Fused (dropout) + residual add + LayerNorm (+ non-pad row mask), forward and backward.
//
//   s   = dropout_p(a[row]) + res[row % res_rows]          (s optionally written back over a)
//   y   = (LN(s) * gamma + beta) * rowscale[row]
//
// This is the post-LN tail of every sub-layer of the reference (modules.py:86-90,117-120), the
// embedding norms (model.py:307-309,433-436: res = positional table, res_rows = T) and the per-block
// `output *= non_pad_mask` (modules.py:154-155,203-204) folded in as rowscale.  HBM-bound: one warp
// per row, 16-byte vector accesses, warp-shuffle statistics, no shared memory.
#include <stdlib.h>
#include "icap_common.cuh"

namespace {

constexpr int MAX_IT = 8;   // d <= MAX_IT * 32 * 4 = 1024 ; kernels are specialised on NIT = ceil(d / 128)

template <int NIT, typename TA, typename TR, typename TY>
__global__ void __launch_bounds__(256)
add_ln_fwd_kernel(int M, int d, TA* __restrict__ a, const TR* __restrict__ res, int res_rows,
                  const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ rowscale,
                  TY* __restrict__ y, float* __restrict__ mean_out, float* __restrict__ rstd_out, int write_sum,
                  float p_drop, uint32_t thresh, uint64_t seed, const int* __restrict__ seed_dev, float eps) {
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int nvec = d >> 2;
  float v[NIT][4];
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  TA* arow = a + (int64_t)row * d;
  const TR* rrow = res ? res + (int64_t)(row % res_rows) * d : nullptr;
  float sum = 0.f;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      load4(arow + vi * 4, v[it]);
      if (p_drop > 0.f) {
        uint32_t keep = dropout_keep4(seed, (uint64_t)row * nvec + vi, thresh);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[it][j] = (keep >> j) & 1 ? v[it][j] * keep_scale : 0.f;
      }
      if (rrow) {
        float r[4];
        load4(rrow + vi * 4, r);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[it][j] += r[j];
      }
      if (write_sum) store4(arow + vi * 4, v[it]);
#pragma unroll
      for (int j = 0; j < 4; ++j) sum += v[it][j];
    }
  }
  const float mean = warp_sum(sum) / (float)d;
  float sq = 0.f;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { float c = v[it][j] - mean; sq += c * c; }
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)d + eps);
  const float rs = rowscale ? rowscale[row] : 1.f;
  TY* yrow = y + (int64_t)row * d;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      float g[4], b[4], o[4];
      load4(gamma + vi * 4, g);
      load4(beta + vi * 4, b);
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = ((v[it][j] - mean) * rstd * g[j] + b[j]) * rs;
      store4(yrow + vi * 4, o);
    }
  }
  if (lane == 0 && mean_out) { mean_out[row] = mean; rstd_out[row] = rstd; }
}

// Backward.  dy = dy1 (+ dy2);  g = dy * rowscale
//   ds = rstd * (g*gamma - mean(g*gamma) - xhat * mean(g*gamma*xhat))      (-> residual branch)
//   da = dropout mask(ds) / (1-p)                                          (-> GEMM branch; == ds if p = 0)
//   dgamma += sum_rows g * xhat ; dbeta += sum_rows g ; dbias2 += sum_rows da
// Two kernels, both streaming at high occupancy: a row kernel (one warp per row, ~60 registers) for ds / da,
// and a column kernel (thread = 2 adjacent columns, rows split over grid.y) for the three column sums.  (A single
// fused kernel needed 180 registers for the per-lane column partials -> 12 % occupancy, 1/5 of HBM speed: ncu r1.)
template <int NIT, typename T>
__global__ void __launch_bounds__(256)
add_ln_bwd_rows_kernel(int M, int d, const T* __restrict__ dy1, const T* __restrict__ dy2, const T* __restrict__ s,
                       const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                       const float* __restrict__ gamma, const float* __restrict__ rowscale, T* __restrict__ ds,
                       T* __restrict__ da, float p_drop, uint32_t thresh, uint64_t seed,
                       const int* __restrict__ seed_dev) {
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int nvec = d >> 2;
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  const float mean = mean_in[row], rstd = rstd_in[row];
  const float rs = rowscale ? rowscale[row] : 1.f;
  float xh[NIT][4], gg[NIT][4];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      float g[4], x[4], gam[4];
      load4(dy1 + (int64_t)row * d + vi * 4, g);
      if (dy2) {
        float g2[4];
        load4(dy2 + (int64_t)row * d + vi * 4, g2);
#pragma unroll
        for (int j = 0; j < 4; ++j) g[j] += g2[j];
      }
      load4(s + (int64_t)row * d + vi * 4, x);
      load4(gamma + vi * 4, gam);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float xhat = (x[j] - mean) * rstd;
        const float gx = g[j] * rs * gam[j];
        xh[it][j] = xhat;
        gg[it][j] = gx;
        s1 += gx;
        s2 += gx * xhat;
      }
    }
  }
  s1 = warp_sum(s1) / (float)d;
  s2 = warp_sum(s2) / (float)d;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = rstd * (gg[it][j] - s1 - xh[it][j] * s2);
      if (ds) store4(ds + (int64_t)row * d + vi * 4, o);
      if (da) {
        if (p_drop > 0.f) {
          uint32_t keep = dropout_keep4(seed, (uint64_t)row * nvec + vi, thresh);
#pragma unroll
          for (int j = 0; j < 4; ++j) o[j] = (keep >> j) & 1 ? o[j] * keep_scale : 0.f;
        }
        store4(da + (int64_t)row * d + vi * 4, o);
      }
    }
  }
}

__device__ __forceinline__ void load2(const float* p, float (&v)[2]) {
  float2 t = *reinterpret_cast<const float2*>(p);
  v[0] = t.x; v[1] = t.y;
}
__device__ __forceinline__ void load2(const bf16* p, float (&v)[2]) {
  __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(p);
  v[0] = __low2float(t); v[1] = __high2float(t);
}

// block (32, 8): 64 columns x 8 row lanes; grid (d/64, row splits)
template <typename T>
__global__ void __launch_bounds__(256)
add_ln_bwd_cols_kernel(int M, int d, const T* __restrict__ dy1, const T* __restrict__ dy2, const T* __restrict__ s,
                       const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                       const float* __restrict__ rowscale, const T* __restrict__ dab, float* __restrict__ dgamma,
                       float* __restrict__ dbeta, float* __restrict__ dbias2, int rows_per_block) {
  pdl_prologue();
  __shared__ float red[3][8][64];
  const int c = blockIdx.x * 64 + threadIdx.x * 2;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float ag[2] = {0.f, 0.f}, ab[2] = {0.f, 0.f}, ac[2] = {0.f, 0.f};
  if (c < d) {
#pragma unroll 4
    for (int r = r0 + threadIdx.y; r < r1; r += 8) {
      float g[2], x[2];
      load2(dy1 + (int64_t)r * d + c, g);
      if (dy2) {
        float g2[2];
        load2(dy2 + (int64_t)r * d + c, g2);
        g[0] += g2[0]; g[1] += g2[1];
      }
      load2(s + (int64_t)r * d + c, x);
      const float mean = mean_in[r], rstd = rstd_in[r], rs = rowscale ? rowscale[r] : 1.f;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float gr = g[j] * rs;
        ag[j] += gr * (x[j] - mean) * rstd;
        ab[j] += gr;
      }
      if (dbias2) {
        float a[2];
        load2(dab + (int64_t)r * d + c, a);
        ac[0] += a[0]; ac[1] += a[1];
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    red[0][threadIdx.y][threadIdx.x * 2 + j] = ag[j];
    red[1][threadIdx.y][threadIdx.x * 2 + j] = ab[j];
    red[2][threadIdx.y][threadIdx.x * 2 + j] = ac[j];
  }
  __syncthreads();
  const int t = threadIdx.y * 32 + threadIdx.x;
  if (t < 192) {
    const int which = t / 64, col = t % 64;
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += red[which][i][col];
    float* dst = which == 0 ? dgamma : which == 1 ? dbeta : dbias2;
    if (dst && blockIdx.x * 64 + col < d) atomicAdd(dst + blockIdx.x * 64 + col, acc);
  }
}


// ------------------------------------------------------------------------------------------------------------
// Fast path (d % 8 == 0, 16-byte aligned rows): 8 elements (16 B of bf16) per lane per access and TWO rows per
// warp, so every warp has 2 x (a, res) [fwd] or 2 x (dy1, dy2, s) [bwd] independent 16-byte loads in flight.
// Dropout indices are element based (e4 = (row*d + col) / 4), i.e. identical to the 4-wide kernels above.
__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const bf16* p, float (&v)[8]) {
  const uint4 t = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(bf16* p, const float (&v)[8]) {
  uint4 t;
  __nv_bfloat162 h;
  h = __floats2bfloat162_rn(v[0], v[1]); t.x = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[2], v[3]); t.y = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[4], v[5]); t.z = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[6], v[7]); t.w = *reinterpret_cast<uint32_t*>(&h);
  *reinterpret_cast<uint4*>(p) = t;
}
__device__ __forceinline__ uint32_t dropout_keep8(uint32_t sf, uint64_t e8, uint32_t thresh) {
  return dropout_keep2(sf, 4 * e8, thresh) | (dropout_keep2(sf, 4 * e8 + 1, thresh) << 2) |
         (dropout_keep2(sf, 4 * e8 + 2, thresh) << 4) | (dropout_keep2(sf, 4 * e8 + 3, thresh) << 6);
}


template <int NIT, int RPW, typename TA, typename TR, typename TY>
__global__ void __launch_bounds__(256)
add_ln_fwd8_kernel(int M, int d, TA* __restrict__ a, const TR* __restrict__ res, int res_rows,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ rowscale,
                   TY* __restrict__ y, float* __restrict__ mean_out, float* __restrict__ rstd_out, int write_sum,
                   float p_drop, uint32_t thresh, uint64_t seed, const int* __restrict__ seed_dev, float eps) {
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  const uint32_t sf = seed_fold(seed);
  const int lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW;
  if (row0 >= M) return;
  const int nvec = d >> 3;
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float v[RPW][NIT][8];
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int row = row0 + r;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int vi = it * 32 + lane;
      if (row < M && vi < nvec) load8(a + (int64_t)row * d + vi * 8, v[r][it]);
    }
  }
  float mean[RPW], rstd[RPW];
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int row = row0 + r;
    const int rrow_i = row < res_rows ? row : row % res_rows;       // residual: usually one row per output row
    const TR* rrow = res ? res + (int64_t)rrow_i * d : nullptr;
    float sum = 0.f;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int vi = it * 32 + lane;
      if (row < M && vi < nvec) {
        if (p_drop > 0.f) {
          dropout_apply8(v[r][it], sf, (uint32_t)row * (uint32_t)nvec + (uint32_t)vi, thresh, keep_scale);
        }
        if (rrow) {
          float rr[8];
          load8(rrow + vi * 8, rr);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[r][it][j] += rr[j];
        }
        if (write_sum) store8(a + (int64_t)row * d + vi * 8, v[r][it]);
#pragma unroll
        for (int j = 0; j < 8; ++j) sum += v[r][it][j];
      }
    }
    mean[r] = warp_sum(sum) / (float)d;
    float sq = 0.f;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int vi = it * 32 + lane;
      if (row < M && vi < nvec) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float c = v[r][it][j] - mean[r]; sq += c * c; }
      }
    }
    rstd[r] = rsqrtf(warp_sum(sq) / (float)d + eps);
  }
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      float g[8], b[8];
      load8(gamma + vi * 8, g);
      load8(beta + vi * 8, b);
#pragma unroll
      for (int r = 0; r < RPW; ++r) {
        const int row = row0 + r;
        if (row < M) {
          const float rs = rowscale ? rowscale[row] : 1.f;
          float o[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = ((v[r][it][j] - mean[r]) * rstd[r] * g[j] + b[j]) * rs;
          store8(y + (int64_t)row * d + vi * 8, o);
        }
      }
    }
  }
  if (lane == 0 && mean_out) {
#pragma unroll
    for (int r = 0; r < RPW; ++r)
      if (row0 + r < M) { mean_out[row0 + r] = mean[r]; rstd_out[row0 + r] = rstd[r]; }
  }
}

template <int NIT, int RPW, typename T>
__global__ void __launch_bounds__(256)
add_ln_bwd_rows8_kernel(int M, int d, const T* __restrict__ dy1, const T* __restrict__ dy2, const T* __restrict__ s,
                        const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                        const float* __restrict__ gamma, const float* __restrict__ rowscale, T* __restrict__ ds,
                        T* __restrict__ da, float p_drop, uint32_t thresh, uint64_t seed,
                        const int* __restrict__ seed_dev) {
  pdl_prologue();
  if (seed_dev) seed += (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull;
  const uint32_t sf = seed_fold(seed);
  const int lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW;
  if (row0 >= M) return;
  const int nvec = d >> 3;
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float xh[RPW][NIT][8], gg[RPW][NIT][8];
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int row = row0 + r;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int vi = it * 32 + lane;
      if (row < M && vi < nvec) {
        load8(dy1 + (int64_t)row * d + vi * 8, gg[r][it]);
        load8(s + (int64_t)row * d + vi * 8, xh[r][it]);
        if (dy2) {
          float g2[8];
          load8(dy2 + (int64_t)row * d + vi * 8, g2);
#pragma unroll
          for (int j = 0; j < 8; ++j) gg[r][it][j] += g2[j];
        }
      }
    }
  }
  float s1[RPW], s2[RPW], rstd[RPW];
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int row = min(row0 + r, M - 1);
    const float mean = mean_in[row], rs = rowscale ? rowscale[row] : 1.f;
    rstd[r] = rstd_in[row];
    float a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int vi = it * 32 + lane;
      if (row0 + r < M && vi < nvec) {
        float gam[8];
        load8(gamma + vi * 8, gam);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xhat = (xh[r][it][j] - mean) * rstd[r];
          const float gx = gg[r][it][j] * rs * gam[j];
          xh[r][it][j] = xhat;
          gg[r][it][j] = gx;
          a1 += gx;
          a2 += gx * xhat;
        }
      }
    }
    s1[r] = warp_sum(a1) / (float)d;
    s2[r] = warp_sum(a2) / (float)d;
  }
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int row = row0 + r;
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int vi = it * 32 + lane;
      if (row < M && vi < nvec) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = rstd[r] * (gg[r][it][j] - s1[r] - xh[r][it][j] * s2[r]);
        if (ds) store8(ds + (int64_t)row * d + vi * 8, o);
        if (da) {
          if (p_drop > 0.f) {
            dropout_apply8(o, sf, (uint32_t)row * (uint32_t)nvec + (uint32_t)vi, thresh, keep_scale);
          }
          store8(da + (int64_t)row * d + vi * 8, o);
        }
      }
    }
  }
}

// block (32, 8): 256 columns (8 per thread, 16-byte loads) x 8 row lanes; grid (d/256, row splits)
template <typename T>
__global__ void __launch_bounds__(256)
add_ln_bwd_cols8_kernel(int M, int d, const T* __restrict__ dy1, const T* __restrict__ dy2, const T* __restrict__ s,
                        const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                        const float* __restrict__ rowscale, const T* __restrict__ dab, float* __restrict__ dgamma,
                        float* __restrict__ dbeta, float* __restrict__ dbias2, int rows_per_block) {
  pdl_prologue();
  __shared__ float red[3][8][256 + 8];
  const int c = blockIdx.x * 256 + threadIdx.x * 8;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float ag[8], ab[8], ac[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ag[j] = 0.f; ab[j] = 0.f; ac[j] = 0.f; }
  if (c < d) {
#pragma unroll 2
    for (int r = r0 + threadIdx.y; r < r1; r += 8) {
      float g[8], x[8];
      load8(dy1 + (int64_t)r * d + c, g);
      load8(s + (int64_t)r * d + c, x);
      if (dy2) {
        float g2[8];
        load8(dy2 + (int64_t)r * d + c, g2);
#pragma unroll
        for (int j = 0; j < 8; ++j) g[j] += g2[j];
      }
      const float mean = mean_in[r], rstd = rstd_in[r], rs = rowscale ? rowscale[r] : 1.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gr = g[j] * rs;
        ag[j] += gr * (x[j] - mean) * rstd;
        ab[j] += gr;
      }
      if (dbias2) {
        float a[8];
        load8(dab + (int64_t)r * d + c, a);
#pragma unroll
        for (int j = 0; j < 8; ++j) ac[j] += a[j];
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[0][threadIdx.y][threadIdx.x * 8 + j] = ag[j];
    red[1][threadIdx.y][threadIdx.x * 8 + j] = ab[j];
    red[2][threadIdx.y][threadIdx.x * 8 + j] = ac[j];
  }
  __syncthreads();
  const int t = threadIdx.y * 32 + threadIdx.x;      // one column per thread, three sums
  if (blockIdx.x * 256 + t < d) {
#pragma unroll
    for (int which = 0; which < 3; ++which) {
      float* dst = which == 0 ? dgamma : which == 1 ? dbeta : dbias2;
      if (!dst) continue;
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) acc += red[which][i][t];
      atomicAdd(dst + blockIdx.x * 256 + t, acc);
    }
  }
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// Start of a KV-cached decode step in ONE launch (was beam_reorder + embed_fwd + add_ln_fwd8: three dependent launches):
// per row (one warp), (1) optionally the beam bookkeeping of the step before -- tokens_out[row, 0..t-1] =
// tokens_in[parent row], tokens_out[row, t] = the chosen token, the same gather on the KV-cache slot table
// (model.py:194-198) -- then (2) y[row] = LayerNorm(table[token] + pos_row) * gamma + beta with exactly the arithmetic of
// embed_fwd_kernel followed by add_ln_fwd8_kernel (decoder input of position t, model.py:432-436), rowscale = token != pad.
template <int NIT, typename T>
__global__ void __launch_bounds__(256)
decode_embed_ln_kernel(int M, int d, int k, int Tmax, int t, const int* __restrict__ parent,
                       const int* __restrict__ token, const int* __restrict__ tok_in, int* __restrict__ tok_out,
                       const int* __restrict__ slot_in, int* __restrict__ slot_out, const T* __restrict__ table,
                       const T* __restrict__ pos_row, const float* __restrict__ gamma, const float* __restrict__ beta,
                       T* __restrict__ y, float* __restrict__ rowscale, int pad, float eps) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  int tk;
  if (parent) {
    const int src = (row / k) * k + parent[row];
    tk = token[row];
    for (int j = lane; j <= t && j < Tmax; j += 32) {
      tok_out[(int64_t)row * Tmax + j] = (j == t) ? tk : tok_in[(int64_t)src * Tmax + j];
      if (slot_in) slot_out[(int64_t)row * Tmax + j] = (j == t) ? row : slot_in[(int64_t)src * Tmax + j];
    }
  } else {
    tk = tok_in[(int64_t)row * Tmax + t];
  }
  const int nvec = d >> 3;
  float v[NIT][8];
  float sum = 0.f;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      load8(table + (int64_t)tk * d + vi * 8, v[it]);
      float rr[8];
      load8(pos_row + vi * 8, rr);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[it][j] += rr[j];
#pragma unroll
      for (int j = 0; j < 8; ++j) sum += v[it][j];
    }
  }
  const float mean = warp_sum(sum) / (float)d;
  float sq = 0.f;
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float c = v[it][j] - mean; sq += c * c; }
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)d + eps);
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int vi = it * 32 + lane;
    if (vi < nvec) {
      float g[8], b[8], o[8];
      load8(gamma + vi * 8, g);
      load8(beta + vi * 8, b);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = ((v[it][j] - mean) * rstd * g[j] + b[j]) * 1.f;
      store8(y + (int64_t)row * d + vi * 8, o);
    }
  }
  if (lane == 0 && rowscale) rowscale[row] = tk != pad ? 1.f : 0.f;
}

}  // namespace

extern "C" int icap_add_ln_fwd(int a_dtype, int act_dtype, int64_t M, int64_t d, void* a, const void* res,
                               int64_t res_rows, const float* gamma, const float* beta, const float* rowscale,
                               void* y, float* mean_out, float* rstd_out, int write_sum, float p_drop,
                               uint64_t seed, const int* seed_dev, float eps, void* stream) {
  ICAP_ARG(d % 4 == 0 && d <= MAX_IT * 128, "icap_add_ln_fwd: d=%lld must be a multiple of 4 and <= %d", (long long)d,
           MAX_IT * 128);
  ICAP_ARG(M > 0 && a && y && gamma && beta, "icap_add_ln_fwd: null argument");
  if (res == nullptr) res_rows = 1;
  ICAP_ARG(res_rows > 0, "icap_add_ln_fwd: res_rows must be positive");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((unsigned)ceil_div64(M, 8));
  const uint32_t th = dropout_threshold(p_drop);
  // go(a element, act element): the three (a, act) combinations that exist; false for any other
  auto by_dtypes = [&](auto go) {
    if (a_dtype == ICAP_F32 && act_dtype == ICAP_F32) go(float{}, float{});
    else if (a_dtype == ICAP_BF16 && act_dtype == ICAP_BF16) go(bf16{}, bf16{});
    else if (a_dtype == ICAP_F32 && act_dtype == ICAP_BF16) go(float{}, bf16{});
    else return false;
    return true;
  };
  bool ok;
  if (d % 8 == 0 && M * (d / 8) < (1ll << 30) && aligned16(a) && aligned16(res) && aligned16(y) && aligned16(gamma) &&
      aligned16(beta) && !env_flag<4>("ICAP_LN_NARROW")) {
    static IcapEnv e_rpw;
    const int rpw = e_rpw.geti("ICAP_LN_RPW", 1);     // rows per warp (1 or 2)
    dim3 grid8((unsigned)ceil_div64(M, 8 * (rpw == 1 ? 1 : 2)));
    ok = by_dtypes([&](auto ta, auto tr) {
      auto go = [&](auto nit, auto r) {
        icap_launch(add_ln_fwd8_kernel<nit, r, decltype(ta), decltype(tr), decltype(tr)>, grid8, 256, 0, st, M, d, a, res,
                    res_rows, gamma, beta, rowscale, y, mean_out, rstd_out, write_sum, p_drop, th, seed, seed_dev, eps);
      };
      auto by_rpw = [&](auto nit) { if (rpw == 1) go(nit, int_c<1>{}); else go(nit, int_c<2>{}); };
      if (d <= 256) by_rpw(int_c<1>{});
      else if (d <= 512) by_rpw(int_c<2>{});
      else by_rpw(int_c<4>{});
    });
  } else {
    ok = by_dtypes([&](auto ta, auto tr) {
      auto go = [&](auto nit) {
        icap_launch(add_ln_fwd_kernel<nit, decltype(ta), decltype(tr), decltype(tr)>, grid, 256, 0, st, M, d, a, res, res_rows,
                    gamma, beta, rowscale, y, mean_out, rstd_out, write_sum, p_drop, th, seed, seed_dev, eps);
      };
      if (d <= 128) go(int_c<1>{});
      else if (d <= 256) go(int_c<2>{});
      else if (d <= 512) go(int_c<4>{});
      else go(int_c<8>{});
    });
  }
  ICAP_ARG(ok, "icap_add_ln_fwd: unsupported dtype combination a=%d act=%d", a_dtype, act_dtype);
  ICAP_LAUNCH_CHECK("icap_add_ln_fwd");
  return 0;
}

// which: bit 0 = row kernel (ds / da), bit 1 = column kernel (dgamma / dbeta / dbias2)
static int add_ln_bwd_impl(int which, int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                           const float* mean, const float* rstd, const float* gamma, const float* rowscale,
                           void* ds, void* da, float* dgamma, float* dbeta, float* dbias2, float p_drop,
                           uint64_t seed, const int* seed_dev, void* stream) {
  ICAP_ARG(d % 4 == 0 && d <= MAX_IT * 128, "icap_add_ln_bwd: d=%lld must be a multiple of 4 and <= %d", (long long)d,
           MAX_IT * 128);
  ICAP_ARG(M > 0 && dy1 && s && mean && rstd && gamma, "icap_add_ln_bwd: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t th = dropout_threshold(p_drop);
  const unsigned row_blocks = (unsigned)ceil_div64(M, 8);
  const int64_t col_blocks = ceil_div64(d, 64);
  int64_t row_splits = ceil_div64(148 * 4, col_blocks);
  if (row_splits > ceil_div64(M, 32)) row_splits = ceil_div64(M, 32);
  const int rows_per_block = (int)ceil_div64(M, row_splits);
  dim3 cgrid((unsigned)col_blocks, (unsigned)ceil_div64(M, rows_per_block)), cblock(32, 8);
  const void* dab = da ? da : ds;       // dbias2 sums the GEMM-branch gradient
  ICAP_ARG(dbias2 == nullptr || dab != nullptr, "icap_add_ln_bwd: dbias2 needs ds or da");
  if (d % 8 == 0 && M * (d / 8) < (1ll << 30) && aligned16(dy1) && aligned16(dy2) && aligned16(s) && aligned16(ds) &&
      aligned16(da) && aligned16(gamma) && !env_flag<4>("ICAP_LN_NARROW")) {
    static IcapEnv e_rpw;
    const int rpw = e_rpw.geti("ICAP_LN_RPW", 1);     // rows per warp (1 or 2)
    const unsigned row_blocks8 = (unsigned)ceil_div64(M, 8 * (rpw == 1 ? 1 : 2));
    const int64_t col_blocks8 = ceil_div64(d, 256);
    static IcapEnv e_cw;
    const int cols_waves = e_cw.geti("ICAP_LN_COLS_WAVES", 3);
    int64_t splits8 = ceil_div64(148 * cols_waves, col_blocks8);
    if (splits8 > ceil_div64(M, 16)) splits8 = ceil_div64(M, 16);
    const int rpb8 = (int)ceil_div64(M, splits8);
    dim3 cgrid8((unsigned)col_blocks8, (unsigned)ceil_div64(M, rpb8));
    dispatch_act(act_dtype, [&](auto tag) {
      using T = decltype(tag);
      if ((ds || da) && (which & 1)) {
        auto go = [&](auto nit, auto r) {
          icap_launch(add_ln_bwd_rows8_kernel<nit, r, T>, row_blocks8, 256, 0, st, M, d, dy1, dy2, s, mean, rstd, gamma,
                      rowscale, ds, da, p_drop, th, seed, seed_dev);
        };
        auto by_rpw = [&](auto nit) { if (rpw == 1) go(nit, int_c<1>{}); else go(nit, int_c<2>{}); };
        if (d <= 256) by_rpw(int_c<1>{});
        else if (d <= 512) by_rpw(int_c<2>{});
        else by_rpw(int_c<4>{});
      }
      if (dgamma || dbeta || dbias2)
        icap_launch(add_ln_bwd_cols8_kernel<T>, cgrid8, cblock, 0, st, M, d, dy1, dy2, s, mean, rstd, rowscale, dab, dgamma,
                    dbeta, dbias2, rpb8);
    });
    ICAP_LAUNCH_CHECK("icap_add_ln_bwd");
    return 0;
  }
  dispatch_act(act_dtype, [&](auto tag) {
    using T = decltype(tag);
    if ((ds || da) && (which & 1)) {
      auto go = [&](auto nit) {
        icap_launch(add_ln_bwd_rows_kernel<nit, T>, row_blocks, 256, 0, st, M, d, dy1, dy2, s, mean, rstd, gamma, rowscale, ds,
                    da, p_drop, th, seed, seed_dev);
      };
      if (d <= 128) go(int_c<1>{});
      else if (d <= 256) go(int_c<2>{});
      else if (d <= 512) go(int_c<4>{});
      else go(int_c<8>{});
    }
    if ((dgamma || dbeta || dbias2) && (which & 2))
      icap_launch(add_ln_bwd_cols_kernel<T>, cgrid, cblock, 0, st, M, d, dy1, dy2, s, mean, rstd, rowscale, dab, dgamma, dbeta,
                  dbias2, rows_per_block);
  });
  ICAP_LAUNCH_CHECK("icap_add_ln_bwd");
  return 0;
}

extern "C" int icap_add_ln_bwd(int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                               const float* mean, const float* rstd, const float* gamma, const float* rowscale,
                               void* ds, void* da, float* dgamma, float* dbeta, float* dbias2, float p_drop,
                               uint64_t seed, const int* seed_dev, void* stream) {
  return add_ln_bwd_impl(3, act_dtype, M, d, dy1, dy2, s, mean, rstd, gamma, rowscale, ds, da, dgamma, dbeta, dbias2,
                         p_drop, seed, seed_dev, stream);
}
// The two halves of icap_add_ln_bwd separately: the parameter-gradient sums (dgamma / dbeta / dbias2) are not on the
// critical path of the backward and may run on another stream AFTER the row kernel has produced ds / da.
extern "C" int icap_add_ln_bwd_rows(int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                                    const float* mean, const float* rstd, const float* gamma, const float* rowscale,
                                    void* ds, void* da, float p_drop, uint64_t seed, const int* seed_dev, void* stream) {
  return add_ln_bwd_impl(1, act_dtype, M, d, dy1, dy2, s, mean, rstd, gamma, rowscale, ds, da, nullptr, nullptr, nullptr,
                         p_drop, seed, seed_dev, stream);
}
extern "C" int icap_add_ln_bwd_params(int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                                      const float* mean, const float* rstd, const float* rowscale, const void* ds,
                                      const void* da, float* dgamma, float* dbeta, float* dbias2, void* stream) {
  alignas(16) static const float dummy_gamma[4] = {0.f, 0.f, 0.f, 0.f};     // not read by the column kernel, only null-checked
  return add_ln_bwd_impl(2, act_dtype, M, d, dy1, dy2, s, mean, rstd, dummy_gamma, rowscale, const_cast<void*>(ds),
                         const_cast<void*>(da), dgamma, dbeta, dbias2, 0.f, 0, nullptr, stream);
}

extern "C" int icap_decode_embed_ln(int act_dtype, int64_t rows, int64_t d, int64_t k, int64_t Tmax, int64_t t,
                                    const int* parent, const int* token, const int* tok_in, int* tok_out,
                                    const int* slot_in, int* slot_out, const void* table, const void* pos_row,
                                    const float* gamma, const float* beta, void* y, float* rowscale, int pad_idx,
                                    float eps, void* stream) {
  ICAP_ARG(rows > 0 && d > 0 && k >= 1 && rows % k == 0 && Tmax > 0 && t >= 0 && t < Tmax && tok_in && table && pos_row &&
           gamma && beta && y, "icap_decode_embed_ln: null/empty argument");
  ICAP_ARG(d % 8 == 0 && d <= 1024 && ((uintptr_t)table & 15) == 0 && ((uintptr_t)pos_row & 15) == 0 &&
           ((uintptr_t)y & 15) == 0 && ((uintptr_t)gamma & 15) == 0 && ((uintptr_t)beta & 15) == 0,
           "icap_decode_embed_ln: width must be a multiple of 8 (<= 1024) and every row pointer 16-byte aligned");
  ICAP_ARG(parent == nullptr || (token && tok_out && tok_out != tok_in && (slot_in == nullptr || (slot_out && slot_out != slot_in))),
           "icap_decode_embed_ln: the beam reorder is out of place and needs token / tok_out (and slot_out with slot_in)");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)ceil_div64(rows, 8);
  dispatch_act(act_dtype, [&](auto tag) {
    auto go = [&](auto nit) {
      icap_launch(decode_embed_ln_kernel<nit, decltype(tag)>, grid, 256, 0, st, rows, d, k, Tmax, t, parent, token, tok_in, tok_out,
                  slot_in, slot_out, table, pos_row, gamma, beta, y, rowscale, pad_idx, eps);
    };
    if (d <= 256) go(int_c<1>{});
    else if (d <= 512) go(int_c<2>{});
    else go(int_c<4>{});
  });
  ICAP_LAUNCH_CHECK("icap_decode_embed_ln");
  return 0;
}
