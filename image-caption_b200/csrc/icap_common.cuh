// Shared device/host helpers for libicap (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#define ICAP_F32 0
#define ICAP_BF16 1

// ---- error plumbing (C ABI: 0 ok, >0 cudaError_t, <0 argument error) -------------------------
void icap_set_error(const char* fmt, ...);

#define ICAP_ARG(cond, ...)                                   \
  do {                                                        \
    if (!(cond)) {                                            \
      icap_set_error(__VA_ARGS__);                            \
      return -1;                                              \
    }                                                         \
  } while (0)

#define ICAP_LAUNCH_CHECK(name)                                               \
  do {                                                                        \
    cudaError_t e__ = cudaGetLastError();                                     \
    if (e__ != cudaSuccess) {                                                 \
      icap_set_error("%s: %s", name, cudaGetErrorString(e__));                \
      return (int)e__;                                                        \
    }                                                                         \
  } while (0)

#define ICAP_CUDA(call)                                                       \
  do {                                                                        \
    cudaError_t e__ = (call);                                                 \
    if (e__ != cudaSuccess) {                                                 \
      icap_set_error("%s: %s", #call, cudaGetErrorString(e__));               \
      return (int)e__;                                                        \
    }                                                                         \
  } while (0)

// ---- launches: every kernel goes through icap_launch so that programmatic dependent launch (PDL) can be
// switched on for the whole library (icap_set_pdl).  Kernels call pdl_wait() before touching global memory
// and pdl_launch_dependents() right after it: the next kernel's CTAs become resident (and run their own
// prologue) while this one is still working, and start the moment this grid has completed and flushed.
extern int icap_g_pdl;
template <typename... KArgs, typename... Args>
static inline cudaError_t icap_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                      Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = icap_g_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() { pdl_wait(); pdl_launch_dependents(); }
#endif

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- environment switches: read ONCE (not per launch); icap_reload_env() (tests / tools that change os.environ in
// the running process) invalidates every cached value.
extern int icap_g_env_gen;
struct IcapEnv {
  int gen = -1;
  const char* v = nullptr;
  const char* get(const char* name) {
    if (gen != icap_g_env_gen) { v = getenv(name); gen = icap_g_env_gen; }
    return v;
  }
  int geti(const char* name, int dflt) { const char* s = get(name); return s ? atoi(s) : dflt; }
};
// is the switch set?  (ID: one cache slot per call-site family; the same ID must always be used with the same name)
template <int ID> static inline bool env_flag(const char* name) {
  static IcapEnv e;
  return e.get(name) != nullptr;
}

// ---- dtype helpers -----------------------------------------------------------------------------
typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(bf16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float x) { return __float2bfloat16_rn(x); }

// 4-wide vector load/store with conversion to/from fp32 (pointer must be 4-element aligned)
__device__ __forceinline__ void load4(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void load4(const bf16* p, float (&v)[4]) {
  uint2 t = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
  v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
}
__device__ __forceinline__ void store4(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void store4(bf16* p, const float (&v)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  uint2 t;
  t.x = *reinterpret_cast<uint32_t*>(&a);
  t.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = t;
}

// ---- warp reductions ----------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- counter-based RNG for dropout ----------------------------------------------------------------
// Stateless: the keep decision of an element is a pure function of (seed, element index), so the backward
// kernels re-evaluate it and no mask tensor is ever stored.  One 32-bit integer hash (lowbias32, two
// multiplies + three xor-shifts) yields two 16-bit uniforms = two elements; an element is kept iff its 16-bit
// uniform >= thresh >> 16.  (Philox4x32-10 here cost ~70 instructions per 4 elements and made the attention
// and LayerNorm kernels issue-bound: ncu r1, profiles/r1_summary.md.)
__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU;
  x ^= x >> 15; x *= 0x846ca68bU;
  x ^= x >> 16;
  return x;
}
__device__ __forceinline__ uint32_t seed_fold(uint64_t seed) {          // loop-invariant: hoisted by the compiler
  return hash32((uint32_t)seed ^ hash32((uint32_t)(seed >> 32) + 0x9E3779B9u));
}
__device__ __forceinline__ uint32_t rand32(uint32_t seed_folded, uint64_t idx) {
  return hash32((uint32_t)idx * 0x9E3779B1u + (uint32_t)(idx >> 32) * 0x85EBCA77u + seed_folded);
}
// keep-mask for the element pair with pair index e2 (elements 2*e2, 2*e2+1): bit j set = keep
__device__ __forceinline__ uint32_t dropout_keep2(uint32_t seed_folded, uint64_t e2, uint32_t thresh) {
  const uint32_t h = rand32(seed_folded, e2), t16 = thresh >> 16;
  return ((h & 0xFFFFu) >= t16 ? 1u : 0u) | ((h >> 16) >= t16 ? 2u : 0u);
}
// keep-mask for 4 consecutive elements starting at element index e4*4
__device__ __forceinline__ uint32_t dropout_keep4(uint64_t seed, uint64_t e4, uint32_t thresh) {
  const uint32_t sf = seed_fold(seed);
  return dropout_keep2(sf, 2 * e4, thresh) | (dropout_keep2(sf, 2 * e4 + 1, thresh) << 2);
}
// v[0..7] = keep ? v * keep_scale : 0 for the 8 elements of vector e8, without materialising the keep mask.
// Same decisions as dropout_keep8 / dropout_keep4 (rand32 of pair index 4*e8 + i; e8 < 2^30 so the index is 32-bit:
// hash32(idx * C + seed) with idx * C advanced by one multiply + adds).
__device__ __forceinline__ void dropout_apply8(float (&v)[8], uint32_t sf, uint32_t e8, uint32_t thresh, float keep_scale) {
  const uint32_t t16 = thresh >> 16;
  uint32_t k = (e8 * 4u) * 0x9E3779B1u + sf;
#pragma unroll
  for (int i = 0; i < 4; ++i, k += 0x9E3779B1u) {
    const uint32_t h = hash32(k);
    v[2 * i] = (h & 0xFFFFu) >= t16 ? v[2 * i] * keep_scale : 0.f;
    v[2 * i + 1] = (h >> 16) >= t16 ? v[2 * i + 1] * keep_scale : 0.f;
  }
}
// Row stride of the attention dropout element index: probability (b, h, i, j) of icap_mha_fwd / icap_mha_bwd is
// element ((b*H + h)*Lq + i) * attn_drop_ld(Lk) + j for every kernel, forward and backward, so a forward on one kernel
// and a backward on another apply the same mask.  For Lk <= 128 it is the key bucket of the mma kernels (16, 32, 48,
// 64, 128; DISPATCH_NT8 picks the kernel from it), above that Lk rounded up to 4.
__host__ __device__ __forceinline__ int attn_drop_ld(int64_t Lk) {
  return Lk <= 16 ? 16 : Lk <= 32 ? 32 : Lk <= 48 ? 48 : Lk <= 64 ? 64 : Lk <= 128 ? 128 : (int)((Lk + 3) & ~3ll);
}
static inline uint32_t dropout_threshold(float p) {
  double t = (double)p * 4294967296.0;
  if (t < 0) t = 0;
  if (t > 4294967295.0) t = 4294967295.0;
  return (uint32_t)t;
}
