// Memory-side kernels of the region feature extractor (the stage BEFORE the caption model: ResNet-101 trunk over the
// 224 x 224 region crops, core/preprocess.py:26-62 -> torchvision resnet101 children[:9]).  Activations are NHWC
// matrices [N*H*W, C] so that every convolution is one icap_gemm (tcgen05 in bf16 mode) over an implicit-GEMM operand:
//   1x1 convolution            : the activation matrix itself (stride 2: a row gather, kh = kw = 1)
//   3x3 / 7x7 convolution      : im2col_nhwc gathers the [N*Ho*Wo, kh*kw*C] patch matrix (zero padding)
//   BatchNorm (+ ReLU, + residual) : the reference never calls .eval() on its extractor (preprocess.py:35-40), so
//                                BatchNorm normalises with the statistics of the batch of crops: bn_stats (per-channel
//                                sum / sum of squares in fp64 atomics) -> bn_finalize (scale, shift, running stats) ->
//                                bn_act (y = relu(x * scale + shift + residual)); eval mode skips the statistics
//   MaxPool 3x3/2, global average pool
// All HBM-bound: 16-byte lanes along C, coalesced rows.
#include "icap_common.cuh"

namespace {

constexpr int NT = 256;

template <typename T> struct Vec8;       // 8 consecutive channels
template <> struct Vec8<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&v)[8]) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
    for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
  }
  static __device__ __forceinline__ void store(bf16* p, const float (&v)[8]) {
    uint4 t;
    __nv_bfloat162 h;
    h = __floats2bfloat162_rn(v[0], v[1]); t.x = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(v[2], v[3]); t.y = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(v[4], v[5]); t.z = *reinterpret_cast<uint32_t*>(&h);
    h = __floats2bfloat162_rn(v[6], v[7]); t.w = *reinterpret_cast<uint32_t*>(&h);
    *reinterpret_cast<uint4*>(p) = t;
  }
};
template <> struct Vec8<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[8]) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
};

// out[(n, ho, wo), (ky, kx, c)] = x[n, ho*s - p + ky, wo*s - p + kx, c]   (0 outside the image; columns >= kh*kw*C zero)
template <typename T>
__global__ void __launch_bounds__(NT)
im2col_kernel(const T* __restrict__ x, int Nimg, int H, int W, int C, int kh, int kw, int stride, int pad, int Ho, int Wo,
              T* __restrict__ out, int64_t ldo, int vec) {
  pdl_prologue();
  const int64_t rows = (int64_t)Nimg * Ho * Wo;
  if (vec) {                                              // C % 8 == 0: one 16-byte (bf16) / 32-byte (fp32) lane per 8 channels
    const int cpr = (int)(ldo / 8), c8 = C / 8;
    const int64_t total = rows * cpr;
    for (int64_t idx = (int64_t)blockIdx.x * NT + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * NT) {
      const int64_t row = idx / cpr;
      const int col8 = (int)(idx - row * cpr);
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const int tap = col8 / c8, cc = (col8 - tap * c8) * 8;
      if (tap < kh * kw) {
        const int wo = (int)(row % Wo), ho = (int)((row / Wo) % Ho), n = (int)(row / ((int64_t)Wo * Ho));
        const int hi = ho * stride - pad + tap / kw, wi = wo * stride - pad + tap % kw;
        if (hi >= 0 && hi < H && wi >= 0 && wi < W) Vec8<T>::load(x + (((int64_t)n * H + hi) * W + wi) * C + cc, v);
      }
      Vec8<T>::store(out + row * ldo + col8 * 8, v);
    }
  } else {
    const int64_t total = rows * ldo;
    const int K = kh * kw * C;
    for (int64_t idx = (int64_t)blockIdx.x * NT + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * NT) {
      const int64_t row = idx / ldo;
      const int col = (int)(idx - row * ldo);
      float v = 0.f;
      if (col < K) {
        const int tap = col / C, c = col - tap * C;
        const int wo = (int)(row % Wo), ho = (int)((row / Wo) % Ho), n = (int)(row / ((int64_t)Wo * Ho));
        const int hi = ho * stride - pad + tap / kw, wi = wo * stride - pad + tap % kw;
        if (hi >= 0 && hi < H && wi >= 0 && wi < W) v = to_f32(x[(((int64_t)n * H + hi) * W + wi) * C + c]);
      }
      out[idx] = from_f32<T>(v);
    }
  }
}

// per-channel sum and sum of squares over M rows (fp64 accumulators: E[x^2] - E[x]^2 without cancellation trouble)
template <typename T>
__global__ void __launch_bounds__(NT)
bn_stats_kernel(const T* __restrict__ x, int64_t M, int C, int64_t ld, double* __restrict__ sums, int rows_per_block) {
  pdl_prologue();
  // thread = 8 channels of one row subset: C / 8 (<= NT) lanes side by side, NT / lanes row subsets per block; the
  // subsets are combined in shared memory so that a block issues one fp64 atomic per channel and statistic
  __shared__ float part[NT][16];
  const int lanes = C / 8, lane = threadIdx.x % lanes, rsub = threadIdx.x / lanes, rstep = NT / lanes;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, q[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int64_t r = r0 + rsub; r < r1; r += rstep) {
    float v[8];
    Vec8<T>::load(x + r * ld + lane * 8, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) { s[i] += v[i]; q[i] = fmaf(v[i], v[i], q[i]); }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) { part[threadIdx.x][i] = s[i]; part[threadIdx.x][8 + i] = q[i]; }
  __syncthreads();
  if (rsub == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a = 0.f, b = 0.f;
      for (int u = 0; u < rstep; ++u) { a += part[u * lanes + lane][i]; b += part[u * lanes + lane][8 + i]; }
      atomicAdd(sums + lane * 8 + i, (double)a);
      atomicAdd(sums + C + lane * 8 + i, (double)b);
    }
  }
}

// scale = gamma * rstd, shift = beta - mean * scale; train mode: batch statistics (biased variance for the
// normalisation, running statistics updated with momentum and the unbiased variance, as nn.BatchNorm2d)
__global__ void bn_finalize_kernel(int C, double* __restrict__ sums, int64_t M, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float momentum, float eps, int train,
                                   float* __restrict__ scale, float* __restrict__ shift) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float mean, var;
  if (train) {
    const double m = sums[c] / (double)M;
    double v = sums[C + c] / (double)M - m * m;
    if (v < 0) v = 0;
    mean = (float)m; var = (float)v;
    if (running_mean) {
      const double unb = M > 1 ? v * (double)M / (double)(M - 1) : v;
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
    }
    sums[c] = 0.0; sums[C + c] = 0.0;                      // ready for the next layer (the buffer is reused)
  } else {
    mean = running_mean[c]; var = running_var[c];
  }
  const float sc = gamma[c] * rsqrtf(var + eps);
  scale[c] = sc;
  shift[c] = beta[c] - mean * sc;
}

template <typename T>
__global__ void __launch_bounds__(NT)
bn_act_kernel(const T* __restrict__ x, int64_t M, int C, const float* __restrict__ scale, const float* __restrict__ shift,
              const T* __restrict__ res, int relu, T* __restrict__ y) {
  pdl_prologue();
  const int c8 = C / 8;
  const int64_t total = M * c8;
  for (int64_t idx = (int64_t)blockIdx.x * NT + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * NT) {
    const int c0 = (int)(idx % c8) * 8;
    float v[8], r[8];
    Vec8<T>::load(x + idx * 8, v);
    if (res) Vec8<T>::load(res + idx * 8, r);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float o = fmaf(v[i], __ldg(scale + c0 + i), __ldg(shift + c0 + i));
      if (res) o += r[i];
      v[i] = relu ? fmaxf(o, 0.f) : o;
    }
    Vec8<T>::store(y + idx * 8, v);
  }
}

template <typename T>
__global__ void __launch_bounds__(NT)
maxpool_kernel(const T* __restrict__ x, int Nimg, int H, int W, int C, int k, int stride, int pad, int Ho, int Wo,
               T* __restrict__ y) {
  pdl_prologue();
  const int c8 = C / 8;
  const int64_t total = (int64_t)Nimg * Ho * Wo * c8;
  for (int64_t idx = (int64_t)blockIdx.x * NT + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * NT) {
    const int c0 = (int)(idx % c8) * 8;
    const int64_t row = idx / c8;
    const int wo = (int)(row % Wo), ho = (int)((row / Wo) % Ho), n = (int)(row / ((int64_t)Wo * Ho));
    float m[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) m[i] = -INFINITY;
    for (int ky = 0; ky < k; ++ky) {
      const int hi = ho * stride - pad + ky;
      if (hi < 0 || hi >= H) continue;
      for (int kx = 0; kx < k; ++kx) {
        const int wi = wo * stride - pad + kx;
        if (wi < 0 || wi >= W) continue;
        float v[8];
        Vec8<T>::load(x + (((int64_t)n * H + hi) * W + wi) * C + c0, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) m[i] = fmaxf(m[i], v[i]);
      }
    }
    Vec8<T>::store(y + row * C + c0, m);
  }
}

// y[n, c] = mean over the HW positions of x[n, :, c]   (fp32 out: the 2048-d region feature)
template <typename T>
__global__ void __launch_bounds__(NT)
avgpool_kernel(const T* __restrict__ x, int HW, int C, float* __restrict__ y) {
  pdl_prologue();
  const int n = blockIdx.y, c8 = C / 8;
  const int g = blockIdx.x * NT + threadIdx.x;
  if (g >= c8) return;
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int p = 0; p < HW; ++p) {
    float v[8];
    Vec8<T>::load(x + ((int64_t)n * HW + p) * C + g * 8, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] += v[i];
  }
  const float inv = 1.f / (float)HW;
#pragma unroll
  for (int i = 0; i < 8; ++i) y[(int64_t)n * C + g * 8 + i] = s[i] * inv;
}

unsigned grid_for(int64_t work_items) {
  int64_t b = ceil_div64(work_items, NT);
  const int64_t cap = 148 * 16;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}
bool al16(const void* p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace

extern "C" int icap_im2col_nhwc(int dtype, const void* x, int64_t N, int64_t H, int64_t W, int64_t C, int kh, int kw,
                                int stride, int pad, void* out, int64_t ldo, void* stream) {
  ICAP_ARG(x && out && N > 0 && H > 0 && W > 0 && C > 0 && kh > 0 && kw > 0 && stride > 0 && pad >= 0, "icap_im2col_nhwc: bad argument");
  const int64_t Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  ICAP_ARG(Ho > 0 && Wo > 0 && ldo >= (int64_t)kh * kw * C, "icap_im2col_nhwc: output too narrow");
  const int vec = (C % 8 == 0 && ldo % 8 == 0 && al16(x) && al16(out)) ? 1 : 0;
  const int64_t work = N * Ho * Wo * (vec ? ldo / 8 : ldo);
  cudaStream_t st = (cudaStream_t)stream;
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(im2col_kernel<decltype(tag)>, grid_for(work), NT, 0, st, x, N, H, W, C, kh, kw, stride, pad, Ho, Wo, out, ldo,
                vec);
  });
  ICAP_LAUNCH_CHECK("icap_im2col_nhwc");
  return 0;
}

extern "C" int icap_bn_scale_shift(int dtype, const void* x, int64_t M, int64_t C, double* sums, const float* gamma,
                                   const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                                   int train, float* scale, float* shift, void* stream) {
  ICAP_ARG(C > 0 && C % 8 == 0 && gamma && beta && scale && shift, "icap_bn_scale_shift: C must be a multiple of 8");
  ICAP_ARG(train ? (x && sums && M > 0 && al16(x)) : (running_mean && running_var), "icap_bn_scale_shift: missing statistics source");
  cudaStream_t st = (cudaStream_t)stream;
  if (train) {
    ICAP_ARG(C / 8 <= NT && NT % (C / 8) == 0, "icap_bn_scale_shift: C / 8 must divide %d", NT);
    const int rows_per_block = 256;
    const unsigned grid = (unsigned)ceil_div64(M, rows_per_block);
    dispatch_act(dtype, [&](auto tag) {
      icap_launch(bn_stats_kernel<decltype(tag)>, grid, NT, 0, st, x, M, C, C, sums, rows_per_block);
    });
    ICAP_LAUNCH_CHECK("icap_bn_scale_shift(stats)");
  }
  icap_launch(bn_finalize_kernel, (unsigned)ceil_div64(C, 128), 128, 0, st, (int)C, sums, M, gamma, beta, running_mean,
              running_var, momentum, eps, train, scale, shift);
  ICAP_LAUNCH_CHECK("icap_bn_scale_shift");
  return 0;
}

extern "C" int icap_bn_act(int dtype, const void* x, int64_t M, int64_t C, const float* scale, const float* shift,
                           const void* residual, int relu, void* y, void* stream) {
  ICAP_ARG(x && y && scale && shift && M > 0 && C > 0 && C % 8 == 0 && al16(x) && al16(y) && al16(residual),
           "icap_bn_act: C must be a multiple of 8 and the tensors 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(bn_act_kernel<decltype(tag)>, grid_for(M * C / 8), NT, 0, st, x, M, C, scale, shift, residual, relu, y);
  });
  ICAP_LAUNCH_CHECK("icap_bn_act");
  return 0;
}

extern "C" int icap_maxpool_nhwc(int dtype, const void* x, int64_t N, int64_t H, int64_t W, int64_t C, int k, int stride,
                                 int pad, void* y, void* stream) {
  ICAP_ARG(x && y && N > 0 && C % 8 == 0 && al16(x) && al16(y), "icap_maxpool_nhwc: C must be a multiple of 8");
  const int64_t Ho = (H + 2 * pad - k) / stride + 1, Wo = (W + 2 * pad - k) / stride + 1;
  cudaStream_t st = (cudaStream_t)stream;
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(maxpool_kernel<decltype(tag)>, grid_for(N * Ho * Wo * C / 8), NT, 0, st, x, N, H, W, C, k, stride, pad, Ho, Wo,
                y);
  });
  ICAP_LAUNCH_CHECK("icap_maxpool_nhwc");
  return 0;
}

extern "C" int icap_avgpool_nhwc(int dtype, const void* x, int64_t N, int64_t HW, int64_t C, float* y, void* stream) {
  ICAP_ARG(x && y && N > 0 && HW > 0 && C % 8 == 0 && al16(x), "icap_avgpool_nhwc: C must be a multiple of 8");
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)ceil_div64(C / 8, NT), (unsigned)N);
  dispatch_act(dtype, [&](auto tag) { icap_launch(avgpool_kernel<decltype(tag)>, grid, NT, 0, st, x, HW, C, y); });
  ICAP_LAUNCH_CHECK("icap_avgpool_nhwc");
  return 0;
}
