// Small HBM-bound kernels around the GEMMs: dtype-converting strided copies (operand packing),
// region-validity masks, caption shifting, embedding gather / scatter-add, column sums (bias grads),
// the fused flat-buffer Adam step, gradient scaling.
#include "icap_common.cuh"
#include <stdarg.h>
#include <string.h>

// --------------------------------------------------------------------------- error string
static thread_local char g_err[512] = "";
void icap_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* icap_last_error() { return g_err; }
int icap_g_pdl = 0;       // launch attribute for every kernel of the library, see icap_launch()
extern "C" int icap_set_pdl(int on) { icap_g_pdl = on ? 1 : 0; return 0; }
int icap_g_env_gen = 0;   // generation of the cached ICAP_* environment switches (IcapEnv, icap_common.cuh)
extern "C" int icap_reload_env(void) { ++icap_g_env_gen; return 0; }

extern "C" int icap_version() { return 100; }

// Refuses to run on anything but Blackwell (sm_100): there is no CPU or other-arch fallback.
extern "C" int icap_sm_check(int device) {
  cudaDeviceProp p;
  ICAP_CUDA(cudaGetDeviceProperties(&p, device));
  ICAP_ARG(p.major == 10, "icap: device %d is sm_%d%d; this library only runs on sm_100a (B200)", device, p.major,
           p.minor);
  return 0;
}

namespace {

template <typename TS, typename TD>
__global__ void copy2d_kernel(const TS* __restrict__ src, int64_t src_ld, TD* __restrict__ dst, int64_t dst_ld,
                              int64_t rows, int64_t cols, int accumulate, int vec) {
  pdl_prologue();
  if (vec) {
    const int64_t c4 = cols >> 2;
    for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < rows * c4; u += (int64_t)gridDim.x * blockDim.x) {
      const int64_t r = u / c4, c = (u % c4) * 4;
      float v[4];
      load4(src + r * src_ld + c, v);
      if (accumulate == 2) {            // atomic: several streams may accumulate into dst concurrently (fp32 dst only)
        if constexpr (sizeof(TD) == 4) {
#pragma unroll
          for (int j = 0; j < 4; ++j) atomicAdd(reinterpret_cast<float*>(dst + r * dst_ld + c) + j, v[j]);
        }
        continue;
      }
      if (accumulate) {
        float o[4];
        load4(dst + r * dst_ld + c, o);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] += o[j];
      }
      store4(dst + r * dst_ld + c, v);
    }
  } else {
    for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < rows * cols; u += (int64_t)gridDim.x * blockDim.x) {
      const int64_t r = u / cols, c = u % cols;
      float v = to_f32(src[r * src_ld + c]);
      if (accumulate == 2) {
        if constexpr (sizeof(TD) == 4) atomicAdd(reinterpret_cast<float*>(dst + r * dst_ld + c), v);
        continue;
      }
      if (accumulate) v += to_f32(dst[r * dst_ld + c]);
      dst[r * dst_ld + c] = from_f32<TD>(v);
    }
  }
}

// a region is padding iff its position row is all zero (model.py:206); one warp per row
__global__ void region_valid_kernel(const float* __restrict__ pos, int64_t M, int Dp, uint8_t* __restrict__ kvalid,
                                    float* __restrict__ rowscale) {
  pdl_prologue();
  const int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  int nz = 0;
  for (int j = lane; j < Dp; j += 32) nz |= (pos[row * Dp + j] != 0.f);
  nz = __any_sync(0xffffffffu, nz);
  if (lane == 0) {
    if (kvalid) kvalid[row] = nz ? 1 : 0;
    if (rowscale) rowscale[row] = nz ? 1.f : 0.f;
  }
}

// region cache -> batch: packed row (b, r) of xcat <- cache row (idx[b], r), with the precomputed validity of that
// region.  One warp per row, 16-byte lanes, 4 loads in flight per lane.  An index outside [0, n_images) raises *err
// and reads image 0 (the output stays defined; the host checks the flag once per epoch).
template <typename TI>
__global__ void gather_regions_kernel(const uint4* __restrict__ cache, const uint8_t* __restrict__ vcache,
                                      const TI* __restrict__ idx, int64_t rows, int R, int row_vec, int64_t n_images,
                                      uint4* __restrict__ xcat, uint8_t* __restrict__ kvalid,
                                      float* __restrict__ rowscale, int* __restrict__ err) {
  pdl_prologue();
  const int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int64_t b = row / R;
  const int r = (int)(row - b * R);
  int64_t img = (int64_t)idx[b];
  if (img < 0 || img >= n_images) {
    if (lane == 0 && err) *err = 1;
    img = 0;
  }
  const uint4* __restrict__ src = cache + (img * R + r) * row_vec;
  uint4* __restrict__ dst = xcat + row * row_vec;
  int j = lane;
  for (; j + 96 < row_vec; j += 128) {
    const uint4 a = __ldg(src + j), c = __ldg(src + j + 32), d = __ldg(src + j + 64), e = __ldg(src + j + 96);
    dst[j] = a; dst[j + 32] = c; dst[j + 64] = d; dst[j + 96] = e;
  }
  for (; j < row_vec; j += 32) dst[j] = __ldg(src + j);
  if (lane == 0) {
    const uint8_t v = vcache[img * R + r];
    kvalid[row] = v;
    rowscale[row] = v ? 1.f : 0.f;
  }
}

// captions [B, L] -> input tokens cap[:, :-1], targets cap[:, 1:], validity, non-pad target count
template <typename TI>
__global__ void caption_prep_kernel(const TI* __restrict__ cap, int B, int L, int pad, int* __restrict__ inp,
                                    int* __restrict__ tgt, uint8_t* __restrict__ tok_valid,
                                    float* __restrict__ rowscale, int* __restrict__ count) {
  pdl_prologue();
  const int T = L - 1;
  int local = 0;
  for (int u = blockIdx.x * blockDim.x + threadIdx.x; u < B * T; u += gridDim.x * blockDim.x) {
    const int b = u / T, t = u % T;
    const int a = (int)cap[(int64_t)b * L + t], n = (int)cap[(int64_t)b * L + t + 1];
    inp[u] = a;
    tgt[u] = n;
    tok_valid[u] = a != pad;
    rowscale[u] = a != pad ? 1.f : 0.f;
    local += (n != pad);
  }
  local = __reduce_add_sync(0xffffffffu, local);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, local);
}

__global__ void count_finish_kernel(const int* __restrict__ count, float* __restrict__ out2) {
  pdl_prologue();
  out2[0] = (float)(*count);
  out2[1] = 1.f / (float)(*count);
}

template <typename TT, typename TO>
__global__ void embed_fwd_kernel(const int* __restrict__ tok, int64_t tok_stride, int64_t M, int E,
                                 const TT* __restrict__ table, TO* __restrict__ out, float* __restrict__ rowscale,
                                 int pad) {
  pdl_prologue();
  const int e4 = E >> 2;
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < M * e4; u += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = u / e4;
    const int c = (int)(u % e4) * 4;
    const int t = tok[r * tok_stride];
    float v[4];
    load4(table + (int64_t)t * E + c, v);
    store4(out + r * E + c, v);
    if (rowscale && c == 0) rowscale[r] = t != pad ? 1.f : 0.f;
  }
}

template <typename T>
__global__ void embed_bwd_kernel(const int* __restrict__ tok, int64_t M, int E, int pad, const T* __restrict__ dout,
                                 float* __restrict__ dtable) {
  pdl_prologue();
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < M * E; u += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = u / E;
    const int c = (int)(u % E);
    const int t = tok[r];
    if (t != pad) atomicAdd(dtable + (int64_t)t * E + c, to_f32(dout[u]));   // padding_idx row keeps zero grad
  }
}

// out[c] += sum_r x[r][c]; block = 32 columns x 8 row-lanes, grid.y splits the rows
template <typename T>
__global__ void colsum_kernel(const T* __restrict__ x, int64_t ld, int64_t M, int64_t N, float* __restrict__ out,
                              int rows_per_block) {
  pdl_prologue();
  __shared__ float red[8][33];
  const int64_t c = blockIdx.x * 32 + threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  const int64_t r1 = min(M, r0 + rows_per_block);
  float s = 0.f;
  if (c < N)
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) s += to_f32(x[r * ld + c]);
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    atomicAdd(out + c, t);
  }
}

// 16-byte variant: thread = 8 adjacent columns, block = 256 columns x 8 row lanes, 2 rows in flight per thread
template <typename T>
__global__ void __launch_bounds__(256)
colsum8_kernel(const T* __restrict__ x, int64_t ld, int64_t M, int64_t N, float* __restrict__ out, int rows_per_block) {
  pdl_prologue();
  __shared__ float red[8][256 + 8];
  const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x * 8;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  const int64_t r1 = min(M, r0 + rows_per_block);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (c < N) {        // N % 8 == 0: a thread's 8 columns are all in range
#pragma unroll 4
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      if constexpr (sizeof(T) == 2) {
        const uint4 t = __ldg(reinterpret_cast<const uint4*>(x + r * ld + c));
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) { acc[2 * i] += __low2float(h[i]); acc[2 * i + 1] += __high2float(h[i]); }
      } else {
        const float4 a = __ldg(reinterpret_cast<const float4*>(x + r * ld + c));
        const float4 b = __ldg(reinterpret_cast<const float4*>(x + r * ld + c) + 1);
        acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
        acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[threadIdx.y][threadIdx.x * 8 + j] = acc[j];
  __syncthreads();
  const int t = threadIdx.y * 32 + threadIdx.x;
  if ((int64_t)blockIdx.x * 256 + t < N) {
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) v += red[i][t];
    atomicAdd(out + (int64_t)blockIdx.x * 256 + t, v);
  }
}

// torch.optim.Adam (no amsgrad, no weight decay), one pass over the flat buffers:
//   m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; p -= (lr / bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
// also refreshes the bf16 shadow copy used by the tensor-core GEMMs.  28 B/param of HBM traffic
// (+2 for the shadow).  step lives on the device so a captured CUDA graph can be replayed.
__global__ void adam_kernel(int64_t n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, bf16* __restrict__ shadow, float lr, float b1, float b2, float eps,
                            const int* __restrict__ step_ptr, const float* __restrict__ gscale_ptr, float gscale,
                            int step_bias) {
  pdl_prologue();
  const int step = *step_ptr + step_bias;
  const float bc1 = 1.f - powf(b1, (float)step);
  const float bc2 = 1.f - powf(b2, (float)step);
  const float step_size = lr / bc1, sqrt_bc2 = sqrtf(bc2);
  const float gs = gscale * (gscale_ptr ? gscale_ptr[0] : 1.f);
  const int64_t n4 = n >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[i], gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    float P[4] = {pp.x, pp.y, pp.z, pp.w}, G[4] = {gg.x, gg.y, gg.z, gg.w};
    float Mm[4] = {mm.x, mm.y, mm.z, mm.w}, Vv[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float gj = G[j] * gs;
      Mm[j] = b1 * Mm[j] + (1.f - b1) * gj;
      Vv[j] = b2 * Vv[j] + (1.f - b2) * gj * gj;
      const float denom = sqrtf(Vv[j]) / sqrt_bc2 + eps;
      P[j] -= step_size * (Mm[j] / denom);
    }
    reinterpret_cast<float4*>(p)[i] = make_float4(P[0], P[1], P[2], P[3]);
    reinterpret_cast<float4*>(m)[i] = make_float4(Mm[0], Mm[1], Mm[2], Mm[3]);
    reinterpret_cast<float4*>(v)[i] = make_float4(Vv[0], Vv[1], Vv[2], Vv[3]);
    if (shadow) store4(shadow + i * 4, P);
  }
}
__global__ void step_tick_kernel(int* step) {
  pdl_prologue(); *step += 1; }
__global__ void reciprocal_kernel(const float* x, float* out, float num) {
  pdl_prologue(); out[0] = num / x[0]; }

__global__ void scale_kernel(float* __restrict__ x, int64_t n, const float* __restrict__ s_ptr, float s) {
  pdl_prologue();
  const float f = s * (s_ptr ? s_ptr[0] : 1.f);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= f;
}

// dst[r][:] = (base ? base[r][:] : 0) + src[(r / div) * mul + off][:]   (row broadcast / gather)
template <typename T>
__global__ void rows_gather_add_kernel(const T* __restrict__ src, int64_t src_ld, const T* __restrict__ base,
                                       int64_t base_ld, T* __restrict__ dst, int64_t dst_ld, int64_t rows, int cols,
                                       int div, int mul, int off) {
  pdl_prologue();
  const int c4 = cols >> 2;
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < rows * c4; u += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = u / c4;
    const int c = (int)(u % c4) * 4;
    float v[4];
    load4(src + ((r / div) * mul + off) * src_ld + c, v);
    if (base) {
      float b[4];
      load4(base + r * base_ld + c, b);
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] += b[j];
    }
    store4(dst + r * dst_ld + c, v);
  }
}
// dst[s * mul + off][:] += sum_{t < seg_len} src[s * seg_len + t][:]       (adjoint of the broadcast)
template <typename T>
__global__ void rows_segsum_add_kernel(const T* __restrict__ src, int64_t src_ld, T* __restrict__ dst, int64_t dst_ld,
                                       int64_t nseg, int seg_len, int cols, int mul, int off) {
  pdl_prologue();
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < nseg * cols; u += (int64_t)gridDim.x * blockDim.x) {
    const int64_t sg = u / cols;
    const int c = (int)(u % cols);
    float acc = 0.f;
    for (int t = 0; t < seg_len; ++t) acc += to_f32(src[(sg * seg_len + t) * src_ld + c]);
    T* d = dst + (sg * mul + off) * dst_ld + c;
    *d = from_f32<T>(to_f32(*d) + acc);
  }
}

inline unsigned grid_for(int64_t work, int threads) {
  int64_t b = ceil_div64(work, threads);
  const int64_t cap = 148 * 16;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

extern "C" int icap_copy2d(const void* src, int src_dtype, int64_t src_ld, void* dst, int dst_dtype, int64_t dst_ld,
                           int64_t rows, int64_t cols, int accumulate, void* stream) {
  ICAP_ARG(src && dst && rows > 0 && cols > 0, "icap_copy2d: null/empty argument");
  ICAP_ARG(accumulate >= 0 && accumulate <= 2 && (accumulate != 2 || dst_dtype == ICAP_F32),
           "icap_copy2d: accumulate must be 0, 1 or 2 (atomic, fp32 destination only)");
  const int ss = src_dtype == ICAP_F32 ? 4 : 2, ds = dst_dtype == ICAP_F32 ? 4 : 2;
  const int vec = (cols % 4 == 0) && ((uintptr_t)src % (4 * ss) == 0) && ((uintptr_t)dst % (4 * ds) == 0) &&
                  (src_ld % 4 == 0) && (dst_ld % 4 == 0);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = grid_for(vec ? rows * cols / 4 : rows * cols, 256);
  auto go = [&](auto ts, auto td) {
    icap_launch(copy2d_kernel<decltype(ts), decltype(td)>, g, 256, 0, st, src, src_ld, dst, dst_ld, rows, cols, accumulate, vec);
  };
  if (src_dtype == ICAP_F32 && dst_dtype == ICAP_F32) go(float{}, float{});
  else if (src_dtype == ICAP_F32 && dst_dtype == ICAP_BF16) go(float{}, bf16{});
  else if (src_dtype == ICAP_BF16 && dst_dtype == ICAP_F32) go(bf16{}, float{});
  else go(bf16{}, bf16{});
  ICAP_LAUNCH_CHECK("icap_copy2d");
  return 0;
}

extern "C" int icap_rows_gather_add(int dtype, const void* src, int64_t src_ld, const void* base, int64_t base_ld,
                                    void* dst, int64_t dst_ld, int64_t rows, int64_t cols, int64_t div, int64_t mul,
                                    int64_t off, void* stream) {
  ICAP_ARG(src && dst && rows > 0 && cols > 0 && cols % 4 == 0 && div > 0, "icap_rows_gather_add: bad argument");
  ICAP_ARG(src_ld % 4 == 0 && dst_ld % 4 == 0 && (base == nullptr || base_ld % 4 == 0),
           "icap_rows_gather_add: leading dimensions must be multiples of 4");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = grid_for(rows * cols / 4, 256);
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(rows_gather_add_kernel<decltype(tag)>, g, 256, 0, st, src, src_ld, base, base_ld, dst, dst_ld, rows, cols, div,
                mul, off);
  });
  ICAP_LAUNCH_CHECK("icap_rows_gather_add");
  return 0;
}

extern "C" int icap_rows_segsum_add(int dtype, const void* src, int64_t src_ld, void* dst, int64_t dst_ld, int64_t nseg,
                                    int64_t seg_len, int64_t cols, int64_t mul, int64_t off, void* stream) {
  ICAP_ARG(src && dst && nseg > 0 && seg_len > 0 && cols > 0, "icap_rows_segsum_add: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = grid_for(nseg * cols, 256);
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(rows_segsum_add_kernel<decltype(tag)>, g, 256, 0, st, src, src_ld, dst, dst_ld, nseg, seg_len, cols, mul, off);
  });
  ICAP_LAUNCH_CHECK("icap_rows_segsum_add");
  return 0;
}

extern "C" int icap_region_valid(const float* pos, int64_t M, int64_t Dp, uint8_t* kvalid, float* rowscale,
                                 void* stream) {
  ICAP_ARG(pos && M > 0 && Dp > 0, "icap_region_valid: null/empty argument");
  icap_launch(region_valid_kernel, (unsigned)ceil_div64(M, 8), 256, 0, (cudaStream_t)stream, pos, M, (int)Dp, kvalid, rowscale);
  ICAP_LAUNCH_CHECK("icap_region_valid");
  return 0;
}

extern "C" int icap_gather_regions(int dtype, const void* cache, const uint8_t* valid_cache, int64_t n_images,
                                   const void* idx, int idx_is_int64, int64_t B, int64_t R, int64_t Kc, void* xcat,
                                   uint8_t* kvalid, float* rowscale, int* err, void* stream) {
  ICAP_ARG(cache && valid_cache && idx && xcat && kvalid && rowscale && n_images > 0 && B > 0 && R > 0 && Kc > 0,
           "icap_gather_regions: null/empty argument");
  ICAP_ARG(dtype == ICAP_F32 || dtype == ICAP_BF16, "icap_gather_regions: dtype must be fp32 or bf16");
  const int64_t row_bytes = Kc * (dtype == ICAP_BF16 ? 2 : 4);
  ICAP_ARG(row_bytes % 16 == 0 && ((uintptr_t)cache & 15) == 0 && ((uintptr_t)xcat & 15) == 0,
           "icap_gather_regions: packed rows must be 16-byte multiples and 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = B * R;
  const unsigned g = (unsigned)ceil_div64(rows, 8);
  auto go = [&](auto ti) {
    icap_launch(gather_regions_kernel<decltype(ti)>, g, 256, 0, st, cache, valid_cache, idx, rows, R, row_bytes / 16,
                n_images, xcat, kvalid, rowscale, err);
  };
  if (idx_is_int64) go(0ll); else go(0);
  ICAP_LAUNCH_CHECK("icap_gather_regions");
  return 0;
}

extern "C" int icap_caption_prep(const void* captions, int cap_is_int64, int64_t B, int64_t L, int pad_idx,
                                 int* inp, int* tgt, uint8_t* tok_valid, float* rowscale, int* count_i,
                                 float* count_f2, void* stream) {
  ICAP_ARG(captions && B > 0 && L > 1 && inp && tgt && tok_valid && rowscale && count_i && count_f2,
           "icap_caption_prep: null/empty argument");
  cudaStream_t st = (cudaStream_t)stream;
  ICAP_CUDA(cudaMemsetAsync(count_i, 0, sizeof(int), st));
  const unsigned g = grid_for(B * (L - 1), 256);
  auto go = [&](auto ti) {
    icap_launch(caption_prep_kernel<decltype(ti)>, g, 256, 0, st, captions, B, L, pad_idx, inp, tgt, tok_valid, rowscale,
                count_i);
  };
  if (cap_is_int64) go(0ll); else go(0);
  icap_launch(count_finish_kernel, 1, 1, 0, st, count_i, count_f2);
  ICAP_LAUNCH_CHECK("icap_caption_prep");
  return 0;
}

extern "C" int icap_embed_fwd(int table_dtype, int out_dtype, const int* tokens, int64_t tok_stride, int64_t M,
                              int64_t E, const void* table, void* out, float* rowscale, int pad_idx, void* stream) {
  ICAP_ARG(tokens && table && out && M > 0 && E % 4 == 0, "icap_embed_fwd: bad argument (E must be a multiple of 4)");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = grid_for(M * E / 4, 256);
  auto go = [&](auto tt, auto to) {
    icap_launch(embed_fwd_kernel<decltype(tt), decltype(to)>, g, 256, 0, st, tokens, tok_stride, M, E, table, out, rowscale,
                pad_idx);
  };
  if (table_dtype == ICAP_F32 && out_dtype == ICAP_F32) go(float{}, float{});
  else if (table_dtype == ICAP_BF16 && out_dtype == ICAP_BF16) go(bf16{}, bf16{});
  else if (table_dtype == ICAP_F32 && out_dtype == ICAP_BF16) go(float{}, bf16{});
  else ICAP_ARG(false, "icap_embed_fwd: unsupported dtype combination");
  ICAP_LAUNCH_CHECK("icap_embed_fwd");
  return 0;
}

extern "C" int icap_embed_bwd(int dtype, const int* tokens, int64_t M, int64_t E, int pad_idx, const void* dout,
                              float* dtable, void* stream) {
  ICAP_ARG(tokens && dout && dtable && M > 0 && E > 0, "icap_embed_bwd: null/empty argument");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = grid_for(M * E, 256);
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(embed_bwd_kernel<decltype(tag)>, g, 256, 0, st, tokens, M, E, pad_idx, dout, dtable);
  });
  ICAP_LAUNCH_CHECK("icap_embed_bwd");
  return 0;
}

extern "C" int icap_colsum(int dtype, int64_t M, int64_t N, const void* x, int64_t ld, float* out, void* stream) {
  ICAP_ARG(x && out && M > 0 && N > 0, "icap_colsum: null/empty argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (N % 8 == 0 && ld % 8 == 0 && ((uintptr_t)x & 15) == 0) {
    const int64_t cb = ceil_div64(N, 256);
    int64_t splits = ceil_div64(148 * 4, cb);
    if (splits > ceil_div64(M, 32)) splits = ceil_div64(M, 32);
    if (splits < 1) splits = 1;
    const int rpb = (int)ceil_div64(M, splits);
    dim3 grid8((unsigned)cb, (unsigned)ceil_div64(M, rpb)), block8(32, 8);
    dispatch_act(dtype, [&](auto tag) { icap_launch(colsum8_kernel<decltype(tag)>, grid8, block8, 0, st, x, ld, M, N, out, rpb); });
    ICAP_LAUNCH_CHECK("icap_colsum");
    return 0;
  }
  const int64_t col_blocks = ceil_div64(N, 32);
  int64_t row_splits = ceil_div64(148 * 8, col_blocks);
  if (row_splits > ceil_div64(M, 64)) row_splits = ceil_div64(M, 64);
  if (row_splits < 1) row_splits = 1;
  const int rows_per_block = (int)ceil_div64(M, row_splits);
  dim3 grid((unsigned)col_blocks, (unsigned)ceil_div64(M, rows_per_block)), block(32, 8);
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(colsum_kernel<decltype(tag)>, grid, block, 0, st, x, ld, M, N, out, rows_per_block);
  });
  ICAP_LAUNCH_CHECK("icap_colsum");
  return 0;
}

extern "C" int icap_adam_step(int64_t n, float* p, const float* g, float* m, float* v, void* shadow_bf16, float lr,
                              float beta1, float beta2, float eps, int* step_dev, int tick, const float* gscale_dev,
                              float gscale, void* stream) {
  ICAP_ARG(n > 0 && n % 4 == 0 && p && g && m && v && step_dev, "icap_adam_step: bad argument (n must be a multiple of 4)");
  cudaStream_t st = (cudaStream_t)stream;
  ICAP_ARG(tick >= 0 && tick <= 2, "icap_adam_step: tick must be 0, 1 or 2");
  if (tick == 1) icap_launch(step_tick_kernel, 1, 1, 0, st, step_dev);
  icap_launch(adam_kernel, grid_for(n / 4, 256), 256, 0, st, n, p, g, m, v, (bf16*)shadow_bf16, lr, beta1, beta2, eps, step_dev,
                                                    gscale_dev, gscale, tick == 2 ? 1 : 0);
  ICAP_LAUNCH_CHECK("icap_adam_step");
  return 0;
}

extern "C" int icap_step_tick(int* step_dev, void* stream) {
  ICAP_ARG(step_dev, "icap_step_tick: null argument");
  icap_launch(step_tick_kernel, 1, 1, 0, (cudaStream_t)stream, step_dev);
  ICAP_LAUNCH_CHECK("icap_step_tick");
  return 0;
}

extern "C" int icap_reciprocal(const float* x, float* out, float numerator, void* stream) {
  ICAP_ARG(x && out, "icap_reciprocal: null argument");
  icap_launch(reciprocal_kernel, 1, 1, 0, (cudaStream_t)stream, x, out, numerator);
  ICAP_LAUNCH_CHECK("icap_reciprocal");
  return 0;
}

extern "C" int icap_scale(float* x, int64_t n, const float* s_dev, float s, void* stream) {
  ICAP_ARG(x && n > 0, "icap_scale: null/empty argument");
  icap_launch(scale_kernel, grid_for(n, 256), 256, 0, (cudaStream_t)stream, x, n, s_dev, s);
  ICAP_LAUNCH_CHECK("icap_scale");
  return 0;
}

// --------------------------------------------------------------------------- GEMM dispatcher

extern "C" int icap_gemm(int ab_dtype, int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, const void* A,
                         int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int c_dtype, const float* bias,
                         int epilogue, const void* aux, int64_t ldaux, int accumulate, int split_k, void* stream) {
  ICAP_ARG(M > 0 && N > 0 && K > 0 && A && B && C, "icap_gemm: null/empty argument");
  ICAP_ARG(epilogue >= 0 && (epilogue & 15) <= 3 && (epilogue & ~31) == 0 && ((epilogue & 15) < 2 || aux),
           "icap_gemm: bad epilogue %d", epilogue);
  ICAP_ARG((epilogue & 15) != 3 || ab_dtype == ICAP_BF16, "icap_gemm: the row-statistics epilogue exists in bf16 mode only");
  ICAP_ARG(accumulate >= 0 && accumulate <= 1, "icap_gemm: accumulate must be 0 or 1");
  ICAP_ARG(M < (1ll << 31) && N < (1ll << 31) && K < (1ll << 31), "icap_gemm: dimension too large");
  cudaStream_t st = (cudaStream_t)stream;
  if (ab_dtype == ICAP_F32) {
    ICAP_ARG(c_dtype == ICAP_F32, "icap_gemm(fp32): C must be fp32");
    return icap_gemm_f32_launch(a_kmajor, b_kmajor, M, N, K, (const float*)A, lda, (const float*)B, ldb, (float*)C, ldc,
                                bias, epilogue & 15, (const float*)aux, ldaux, accumulate, split_k, st);
  }
  return icap_gemm_bf16_launch(a_kmajor, b_kmajor, M, N, K, A, lda, B, ldb, C, ldc, c_dtype, bias, epilogue, aux, ldaux,
                               accumulate, split_k, st);
}
