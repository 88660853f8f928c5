// Vocabulary-side kernels: fused log-softmax + NLL (+ in-place dlogits), loss finalisation
// (mean over non-pad targets, optional focal transform), greedy argmax, and the beam-search
// candidate selection (softmax + running score + top-k over k*V + parent/token split).
//
// Reference semantics:
//   CrossEntropyLoss(ignore_index=pad, reduction='mean')                 model.py:76,93-96
//   FocalLoss: ce scalar -> (1 - exp(-ce))^2 * ce                        loss.py:20-28
//   greedy: argmax(Softmax(logits))                                      model.py:125-128
//   beam  : Softmax(logits) + prev_score, cat over beams, topk(k),
//           parent = idx // V, token = idx % V                           model.py:181-198
//           (LogSoftmax in the PolicyNetwork variant, model_RL.py:72)
// Not in the reference: the <END>-aware variant of the beam step (EOS template flag of the beam_select kernels; finished
// hypotheses carry their score unchanged) and the final length-normalised ranking of the beams (beam_finalize_kernel).
#include "icap_common.cuh"

namespace {

constexpr int NT = 256;

__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
  for (int i = 1; i < NT / 32; ++i) r = fmaxf(r, red[i]);
  return r;
}
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int i = 0; i < NT / 32; ++i) r += red[i];   // fixed order: deterministic
  return r;
}

// one block per row; the row is staged once in shared memory as fp32 when it fits
template <typename T>
__global__ void __launch_bounds__(NT)
xent_kernel(int V, T* __restrict__ logits, int64_t ldl, const int* __restrict__ targets, int ignore_index,
            const float* __restrict__ inv_count, float* __restrict__ row_loss, int write_grad, int cached, int vec) {
  pdl_prologue();
  extern __shared__ __align__(16) float xs[];
  __shared__ float red[NT / 32];
  const int row = blockIdx.x;
  T* x = logits + (int64_t)row * ldl;
  const int tgt = targets[row];
  const bool valid = tgt != ignore_index;
  if (!valid && !write_grad) {
    if (threadIdx.x == 0) row_loss[row] = 0.f;
    return;
  }
  float mx = -INFINITY;
  const int V4 = vec ? (V & ~3) : 0;
  for (int j = threadIdx.x * 4; j < V4; j += NT * 4) {
    float v[4];
    load4(x + j, v);
    if (cached) *reinterpret_cast<float4*>(xs + j) = make_float4(v[0], v[1], v[2], v[3]);
    mx = fmaxf(fmaxf(mx, fmaxf(v[0], v[1])), fmaxf(v[2], v[3]));
  }
  for (int j = V4 + threadIdx.x; j < V; j += NT) {
    const float v = to_f32(x[j]);
    if (cached) xs[j] = v;
    mx = fmaxf(mx, v);
  }
  mx = block_max(mx, red);
  // bf16 logits carry 8 bits: the approximate exponential (2 ulp of fp32) is far below their rounding; fp32 mode keeps expf
  constexpr bool kFastExp = sizeof(T) == 2;
  const float x_tgt = valid ? to_f32(x[tgt]) : 0.f;            // read before the gradients overwrite the row
  float sum = 0.f;
  if (cached) {
    // the row sits in shared memory: replace every logit by exp(x - max) once; the gradient pass only scales it
    for (int j = threadIdx.x; j < V; j += NT) {
      const float e = kFastExp ? __expf(xs[j] - mx) : expf(xs[j] - mx);
      xs[j] = e;
      sum += e;
    }
  } else {
    for (int j = threadIdx.x; j < V; j += NT) sum += kFastExp ? __expf(to_f32(x[j]) - mx) : expf(to_f32(x[j]) - mx);
  }
  sum = block_sum(sum, red);
  const float lse = mx + logf(sum);
  if (threadIdx.x == 0) row_loss[row] = valid ? lse - x_tgt : 0.f;
  if (write_grad) {
    const float sc = valid ? *inv_count : 0.f;
    const float inv_sum = 1.f / sum;
    for (int j = threadIdx.x * 4; j < V4; j += NT * 4) {
      float g[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float pr = cached ? xs[j + t] * inv_sum
                                : (kFastExp ? __expf(to_f32(x[j + t]) - lse) : expf(to_f32(x[j + t]) - lse));
        g[t] = (pr - ((j + t) == tgt ? 1.f : 0.f)) * sc;
      }
      store4(x + j, g);
    }
    for (int j = V4 + threadIdx.x; j < V; j += NT) {
      const float pr = cached ? xs[j] * inv_sum : (kFastExp ? __expf(to_f32(x[j]) - lse) : expf(to_f32(x[j]) - lse));
      x[j] = from_f32<T>((pr - (j == tgt ? 1.f : 0.f)) * sc);
    }
  }
}

// The same loss / gradient with the whole row in REGISTERS (bf16 logits, V <= NV * 2048, V % 8 == 0, 16-byte aligned rows):
// one 16-byte load and one 16-byte store per 8 logits and no shared-memory round trips -- the shared-memory version above
// spends 72 % of its issue slots on 155 MB of traffic (profiles/r2_summary.md section 3).
template <int NV>
__global__ void __launch_bounds__(NT)
xent_reg_kernel(int V, bf16* __restrict__ logits, int64_t ldl, const int* __restrict__ targets, int ignore_index,
                const float* __restrict__ inv_count, float* __restrict__ row_loss, int write_grad) {
  pdl_prologue();
  __shared__ float red[NT / 32];
  const int row = blockIdx.x;
  bf16* x = logits + (int64_t)row * ldl;
  const int tgt = targets[row];
  const bool valid = tgt != ignore_index;
  if (!valid && !write_grad) {
    if (threadIdx.x == 0) row_loss[row] = 0.f;
    return;
  }
  float v[NV][8];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int j = (i * NT + threadIdx.x) * 8;
    if (j < V) {
      const uint4 t = *reinterpret_cast<const uint4*>(x + j);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
      for (int e = 0; e < 4; ++e) { v[i][2 * e] = __low2float(h[e]); v[i][2 * e + 1] = __high2float(h[e]); }
#pragma unroll
      for (int e = 0; e < 8; ++e) mx = fmaxf(mx, v[i][e]);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[i][e] = -INFINITY;
    }
  }
  const float x_tgt = valid ? to_f32(x[tgt]) : 0.f;             // read before any thread overwrites the row (barriers below)
  mx = block_max(mx, red);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { v[i][e] = __expf(v[i][e] - mx); sum += v[i][e]; }
  }
  sum = block_sum(sum, red);
  if (threadIdx.x == 0) row_loss[row] = valid ? mx + logf(sum) - x_tgt : 0.f;
  if (write_grad) {
    const float sc = valid ? *inv_count : 0.f, inv_sum = 1.f / sum;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int j = (i * NT + threadIdx.x) * 8;
      if (j < V) {
        uint4 t;
        uint32_t* w = reinterpret_cast<uint32_t*>(&t);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float g0 = (v[i][2 * e] * inv_sum - (j + 2 * e == tgt ? 1.f : 0.f)) * sc;
          const float g1 = (v[i][2 * e + 1] * inv_sum - (j + 2 * e + 1 == tgt ? 1.f : 0.f)) * sc;
          const __nv_bfloat162 hh = __floats2bfloat162_rn(g0, g1);
          w[e] = *reinterpret_cast<const uint32_t*>(&hh);
        }
        *reinterpret_cast<uint4*>(x + j) = t;
      }
    }
  }
}

__global__ void __launch_bounds__(NT)
xent_finalize_kernel(int M, const float* __restrict__ row_loss, const float* __restrict__ inv_count, int focal,
                     float* __restrict__ out) {
  pdl_prologue();
  __shared__ float red[NT / 32];
  float s = 0.f;
  for (int i = threadIdx.x; i < M; i += NT) s += row_loss[i];
  s = block_sum(s, red);
  if (threadIdx.x == 0) {
    const float ce = s * (*inv_count);
    if (focal) {
      const float pt = expf(-ce), om = 1.f - pt;
      out[0] = om * om * ce;
      out[1] = 2.f * om * pt * ce + om * om;   // d focal / d ce : scales every gradient
    } else {
      out[0] = ce;
      out[1] = 1.f;
    }
  }
}

// up to 8 consecutive logits starting at x[j] as fp32 (one 16-byte load when `vec` and all 8 are in range)
template <typename T>
__device__ __forceinline__ int load_chunk8(const T* __restrict__ x, int j, int V, bool vec, float (&v)[8]) {
  const int n = min(8, V - j);
  if (vec && n == 8) {
    if constexpr (sizeof(T) == 2) {
      const uint4 t = *reinterpret_cast<const uint4*>(x + j);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
      for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
    } else {
      const float4 a = *reinterpret_cast<const float4*>(x + j), b = *reinterpret_cast<const float4*>(x + j + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = i < n ? to_f32(x[j + i]) : -INFINITY;
  }
  return n;
}


template <typename T>
__global__ void __launch_bounds__(NT)
argmax_kernel(int V, const T* __restrict__ logits, int64_t ldl, int* __restrict__ out, int64_t out_stride,
              float* __restrict__ gap) {
  pdl_prologue();
  __shared__ float sv[NT], sv2[NT];
  __shared__ int si[NT];
  const T* x = logits + (int64_t)blockIdx.x * ldl;
  float best = -INFINITY, second = -INFINITY;
  int bi = 0x7fffffff;
  const bool vec = ((uintptr_t)logits % 16 == 0) && (ldl * sizeof(T)) % 16 == 0;
  for (int j0 = threadIdx.x * 8; j0 < V; j0 += NT * 8) {       // ascending index per thread: first maximum is kept
    float c[8];
    const int n = load_chunk8(x, j0, V, vec, c);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i >= n) break;
      const float v = c[i];
      if (v > best) { second = best; best = v; bi = j0 + i; }
      else if (v > second) second = v;
    }
  }
  sv[threadIdx.x] = best; sv2[threadIdx.x] = second; si[threadIdx.x] = bi;
  __syncthreads();
  for (int s = NT / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      const float a = sv[threadIdx.x], b = sv[threadIdx.x + s];
      const int ia = si[threadIdx.x], ib = si[threadIdx.x + s];
      const float a2 = sv2[threadIdx.x], b2 = sv2[threadIdx.x + s];
      if (b > a || (b == a && ib < ia)) {       // lowest index wins ties (torch.argmax on CPU)
        sv[threadIdx.x] = b; si[threadIdx.x] = ib; sv2[threadIdx.x] = fmaxf(a, b2);
      } else {
        sv2[threadIdx.x] = fmaxf(a2, b);
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[(int64_t)blockIdx.x * out_stride] = si[0];
    if (gap) gap[blockIdx.x] = sv[0] - sv2[0];
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Sampled decoding step (icap_sample_tokens): one block per row, inverse-CDF draw from p_j ~ exp((x_j - max) / tau) and
// the tau = 1 log-probability of the drawn token.  Thread i owns the contiguous columns [i*per, (i+1)*per) (per = a
// multiple of 8, so its loads are 16-byte vectors), which fixes the order of the running sum: the running sum at column j
// of chunk i is fl(P_i + L_j), P_i the block's exclusive scan of the chunk sums and L_j the chunk's own sequential sum up
// to j.  It is non-decreasing inside a chunk and ends at fl(P_i + c_i), so the first chunk whose end exceeds u * sum
// holds the token, and only its thread walks its columns a second time.
__device__ __forceinline__ float sample_weight(float v, float mx, float inv_tau, bool tau_one) {
  return tau_one ? expf(v - mx) : expf((v - mx) * inv_tau);
}

template <typename T>
__global__ void __launch_bounds__(NT)
sample_kernel(int V, const T* __restrict__ logits, int64_t ldl, float inv_tau, uint64_t seed,
              const int* __restrict__ seed_dev, int t, int Tmax, int* __restrict__ tokens, float* __restrict__ logp,
              int64_t ldp, int end_idx, int pad_idx) {
  pdl_prologue();                                   // the classifier GEMM writes the logits: nothing is read before
  __shared__ float red[NT / 32];
  __shared__ float s_wsum[NT / 32];
  __shared__ unsigned s_flag[NT / 32];
  __shared__ int s_last[NT / 32];
  __shared__ int s_tok;
  const int row = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int* tok = tokens + (int64_t)row * Tmax;
  float* lp = logp + (int64_t)row * ldp + t;
  if (t >= 1) {                                     // finished row (the StructureCriterion mask rule): pad, log-prob 0
    const int prev = tok[t];
    if (prev == end_idx || prev == pad_idx) {
      if (threadIdx.x == 0) { tok[t + 1] = pad_idx; *lp = 0.f; }
      return;
    }
  }
  const T* x = logits + (int64_t)row * ldl;
  const bool vec = ((uintptr_t)logits % 16 == 0) && (ldl * sizeof(T)) % 16 == 0;
  const int per = ((V + 7) / 8 + NT - 1) / NT * 8;
  const int jb = min(threadIdx.x * per, V), je = min(jb + per, V);
  float mx = -INFINITY;
  for (int j = jb; j < je; j += 8) {
    float c[8];
    load_chunk8(x, j, V, vec, c);                   // columns >= V read as -inf
#pragma unroll
    for (int i = 0; i < 8; ++i) mx = fmaxf(mx, c[i]);
  }
  mx = block_max(mx, red);
  const bool tau_one = inv_tau == 1.f;
  float csum = 0.f, s1 = 0.f;                       // chunk sum of the tempered weights; sum of exp(x - max)
  int last = -1;                                    // last column of the chunk with a non-zero weight
  for (int j = jb; j < je; j += 8) {
    float c[8];
    const int n = load_chunk8(x, j, V, vec, c);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i >= n) break;
      const float e = expf(c[i] - mx);
      const float w = tau_one ? e : sample_weight(c[i], mx, inv_tau, false);
      csum += w;
      s1 += e;
      if (w > 0.f) last = j + i;
    }
  }
  // exclusive scan of the chunk sums (fixed order), the total, and the sum of exp(x - max)
  float incl = csum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  float excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = 0.f;
  const int wlast = __reduce_max_sync(0xffffffffu, last + 1) - 1;
  if (lane == 31) s_wsum[warp] = incl;
  if (lane == 0) s_last[warp] = wlast;
  s1 = block_sum(s1, red);                          // its barriers also publish s_wsum / s_last
  float pre = 0.f, total = 0.f;
  int glast = -1;
  for (int w = 0; w < NT / 32; ++w) {
    if (w < warp) pre += s_wsum[w];
    total += s_wsum[w];
    glast = max(glast, s_last[w]);
  }
  const float P = pre + excl;
  // u in (0, 1) with 24 random bits; u * total is exact in double, and so is every comparison with it
  const uint64_t es = seed + (seed_dev ? (uint64_t)(*seed_dev) * 0x9E3779B97F4A7C15ull : 0ull);
  const uint32_t h = rand32(seed_fold(es), (uint64_t)row * Tmax + t);
  const double target = ((double)(h >> 8) + 0.5) * 0x1p-24 * (double)total;
  const bool flag = csum > 0.f && (double)(P + csum) > target;
  const unsigned ball = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) s_flag[warp] = ball;
  __syncthreads();
  int owner = -1;
  for (int w = 0; w < NT / 32; ++w) {
    if (s_flag[w]) { owner = w * 32 + __ffs(s_flag[w]) - 1; break; }
  }
  if (owner < 0) {                                  // rounding left no column above u * sum: the last non-zero weight
    if (threadIdx.x == 0) s_tok = glast >= 0 ? glast : 0;
  } else if ((int)threadIdx.x == owner) {
    float L = 0.f;
    int pick = -1;
    for (int j = jb; j < je && pick < 0; j += 8) {
      float c[8];
      const int n = load_chunk8(x, j, V, vec, c);
      for (int i = 0; i < n; ++i) {
        L += sample_weight(c[i], mx, inv_tau, tau_one);
        if ((double)(P + L) > target) { pick = j + i; break; }
      }
    }
    s_tok = pick >= 0 ? pick : last;                // not reached: the chunk's end exceeds the target
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int k = s_tok;
    tok[t + 1] = k;
    *lp = (float)((double)to_f32(x[k]) - (double)mx - log((double)s1));
  }
}

constexpr int CAND_CAP = 1024;   // fast-path candidate list of beam_select
constexpr int KMAX = 8;   // beam width limit; lists hold KMAX+1 entries so the k/(k+1) gap can be reported

struct Cand { float s; int i; };
__device__ __forceinline__ bool better(float s, int i, float s2, int i2) { return s > s2 || (s == s2 && i < i2); }

// End-of-sequence handling of icap_beam_select_eos: hypothesis `row` is finished at step t >= 1 when its token at
// position t is end_idx or pad_idx (the rule of icap_sample_tokens); a finished row offers the one candidate
// (token pad_idx, score prev[row]) instead of its V logits.
struct EosArgs {
  const int* tokens;
  int Tmax, t, end_idx, pad_idx;
};
__device__ __forceinline__ bool eos_finished(const EosArgs& e, int row) {
  if (e.t < 1) return false;
  const int tk = e.tokens[(int64_t)row * e.Tmax + e.t];
  return tk == e.end_idx || tk == e.pad_idx;
}

// Exact selection without a candidate bound: every thread keeps the sorted best L of the candidates it scans, the block
// merges the lists.  The fall-back of both beam_select kernels when more than CAND_CAP candidates tie with the bound
// (degenerate logits); needs the softmax maximum / denominator of every row in s_mx / s_den.  Whole block, convergent.
// EOS: rows with s_fin[r] set scan nothing; thread 0 offers their single candidate (prev, r * V + pad_idx).
template <typename T, bool EOS = false>
__device__ __forceinline__ void beam_select_exact(int b, int kin, int V, const T* __restrict__ logits, int64_t ldl,
                                               const float* __restrict__ prev, int kout, float* __restrict__ out_score,
                                               int* __restrict__ out_parent, int* __restrict__ out_token,
                                               float* __restrict__ gap, int log_domain, const float* s_mx,
                                               const float* s_den, float* h_s, int* h_i, int* h_t,
                                               const int* s_fin = nullptr, int pad_idx = 0) {
  const bool vec = ((uintptr_t)logits % 16 == 0) && (ldl * sizeof(T)) % 16 == 0;
  const int L = kout + 1;
  Cand lst[KMAX + 1];                      // sorted, best first; only static indices (stays in registers)
#pragma unroll
  for (int t = 0; t <= KMAX; ++t) { lst[t].s = -INFINITY; lst[t].i = 0x7fffffff; }
  float worst_s = -INFINITY;               // == lst[L-1]: the entry a candidate has to beat
  int worst_i = 0x7fffffff;
  auto push = [&](float sc, int idx) {     // sc, idx beat (worst_s, worst_i): insert, keep the list sorted
#pragma unroll
    for (int t = 0; t <= KMAX; ++t) if (t == L - 1) { lst[t].s = sc; lst[t].i = idx; }
#pragma unroll
    for (int t = KMAX; t > 0; --t) {
      if (t < L && better(lst[t].s, lst[t].i, lst[t - 1].s, lst[t - 1].i)) {
        Cand c = lst[t]; lst[t] = lst[t - 1]; lst[t - 1] = c;
      }
    }
#pragma unroll
    for (int t = 0; t <= KMAX; ++t) if (t == L - 1) { worst_s = lst[t].s; worst_i = lst[t].i; }
  };
  for (int r = 0; r < kin; ++r) {
    if constexpr (EOS) {
      if (s_fin[r]) {
        const float pv = prev ? prev[b * kin + r] : 0.f;
        if (threadIdx.x == 0 && better(pv, r * V + pad_idx, worst_s, worst_i)) push(pv, r * V + pad_idx);
        continue;
      }
    }
    const T* x = logits + ((int64_t)b * kin + r) * ldl;
    const float mx = s_mx[r], den = s_den[r], pv = prev ? prev[b * kin + r] : 0.f;
    // Cheap pre-filter in the logit domain: the score is monotonic in the logit, so only logits above
    //   tl = logit whose score equals the current worst list entry (minus a 1e-3 safety margin)
    // can enter the list; everything else costs one compare instead of expf + divide.
    float tl;
    auto refresh_tl = [&]() {
      if (log_domain) tl = worst_s - pv + mx + den;
      else { const float need = worst_s - pv; tl = need > 0.f ? mx + logf(need * den) : -INFINITY; }
      tl -= 1e-3f;
    };
    refresh_tl();
    for (int j0 = threadIdx.x * 8; j0 < V; j0 += NT * 8) {
      float v[8];
      const int n = load_chunk8(x, j0, V, vec, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i >= n) break;
        const float xv = v[i];
        if (!(xv > tl)) continue;
        const float sc = (log_domain ? (xv - mx - den) : (expf(xv - mx) / den)) + pv;
        const int idx = r * V + j0 + i;
        if (better(sc, idx, worst_s, worst_i)) {
          push(sc, idx);
          refresh_tl();
        }
      }
    }
  }
  // block merge: L rounds of "best remaining head"
  int head = 0;
  float kth = 0.f;
  for (int round = 0; round < L; ++round) {
    float hs = -INFINITY;
    int hi = 0x7fffffff;
#pragma unroll
    for (int t = 0; t <= KMAX; ++t) if (t == head && t < L) { hs = lst[t].s; hi = lst[t].i; }
    h_s[threadIdx.x] = hs;
    h_i[threadIdx.x] = hi;
    h_t[threadIdx.x] = threadIdx.x;
    __syncthreads();
    for (int s = NT / 2; s > 0; s >>= 1) {
      if (threadIdx.x < s) {
        if (better(h_s[threadIdx.x + s], h_i[threadIdx.x + s], h_s[threadIdx.x], h_i[threadIdx.x])) {
          h_s[threadIdx.x] = h_s[threadIdx.x + s];
          h_i[threadIdx.x] = h_i[threadIdx.x + s];
          h_t[threadIdx.x] = h_t[threadIdx.x + s];
        }
      }
      __syncthreads();
    }
    const int winner = h_t[0];
    const float ws = h_s[0];
    const int wi = h_i[0];
    if (threadIdx.x == winner) ++head;
    if (threadIdx.x == 0) {
      if (round < kout) {
        out_score[b * kout + round] = ws;
        out_parent[b * kout + round] = wi / V;
        out_token[b * kout + round] = wi % V;
        kth = ws;
      } else if (gap) {
        gap[b] = kth - ws;
      }
    }
    __syncthreads();
  }
}

template <typename T, bool EOS = false>
__global__ void __launch_bounds__(NT)
beam_select_kernel(int kin, int V, const T* __restrict__ logits, int64_t ldl, const float* __restrict__ prev,
                   int kout, float* __restrict__ out_score, int* __restrict__ out_parent, int* __restrict__ out_token,
                   float* __restrict__ gap, int log_domain, EosArgs eos) {
  pdl_prologue();
  __shared__ float red[NT / 32];
  __shared__ float s_mx[KMAX], s_den[KMAX];
  __shared__ float h_s[NT];
  __shared__ int h_i[NT], h_t[NT];
  const int b = blockIdx.x;
  const bool vec = ((uintptr_t)logits % 16 == 0) && (ldl * sizeof(T)) % 16 == 0;
  const int L = kout + 1;
  __shared__ float s_w1[KMAX][NT / 32], s_w2[KMAX][NT / 32];   // two largest logits of every (row, warp)
  __shared__ float s_we[KMAX][NT / 32];
  __shared__ float c_s[CAND_CAP];
  __shared__ int c_i[CAND_CAP];
  __shared__ int c_n;
  __shared__ float s_tau;
  __shared__ int s_fin[KMAX];                         // EOS: row r is finished
  if constexpr (EOS) {
    if (threadIdx.x < kin) s_fin[threadIdx.x] = eos_finished(eos, b * kin + threadIdx.x);
    __syncthreads();
  }
  for (int r = 0; r < kin; ++r) {
    if constexpr (EOS) {
      if (s_fin[r]) {                                 // no logits read: the row's statistics stay empty
        if ((threadIdx.x & 31) == 0) {
          s_w1[r][threadIdx.x >> 5] = -INFINITY; s_w2[r][threadIdx.x >> 5] = -INFINITY; s_we[r][threadIdx.x >> 5] = 0.f;
        }
        continue;
      }
    }
    const T* x = logits + ((int64_t)b * kin + r) * ldl;
    // ONE pass: the thread's two largest logits (t1 >= t2) and its online softmax sum  es = sum exp(x - t1)
    float t1 = -INFINITY, t2 = -INFINITY, es = 0.f;
    for (int j = threadIdx.x * 8; j < V; j += NT * 8) {
      float v[8];
      load_chunk8(x, j, V, vec, v);                   // out-of-range elements arrive as -inf
      const float old = t1;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float xv = v[i];
        if (xv > t1) { t2 = t1; t1 = xv; } else if (xv > t2) t2 = xv;
      }
      if (t1 > old) es *= expf(old - t1);             // new running maximum: rescale what has been summed
      if (t1 > -INFINITY) {
#pragma unroll
        for (int i = 0; i < 8; ++i) es += expf(v[i] - t1);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {                // merge the sorted pairs and the (max, sum) pairs across the warp
      const float o1 = __shfl_xor_sync(0xffffffffu, t1, o), o2 = __shfl_xor_sync(0xffffffffu, t2, o);
      const float oe = __shfl_xor_sync(0xffffffffu, es, o);
      const float n1 = fmaxf(t1, o1);
      es = es * (t1 == n1 ? 1.f : expf(t1 - n1)) + oe * (o1 == n1 ? 1.f : expf(o1 - n1));
      t2 = fmaxf(fminf(t1, o1), fmaxf(t2, o2));
      t1 = n1;
    }
    if ((threadIdx.x & 31) == 0) {                    // per-(row, warp) slots: no block barrier between the rows
      s_w1[r][threadIdx.x >> 5] = t1; s_w2[r][threadIdx.x >> 5] = t2;      // this warp's two largest logits of row r
      s_we[r][threadIdx.x >> 5] = es;                                      // and its sum of exp(x - t1)
    }
  }
  if (threadIdx.x == 0) c_n = 0;
  __syncthreads();
  if (threadIdx.x < kin) {                            // thread r: softmax maximum and denominator of row r
    const int r = threadIdx.x;
    float mx = s_w1[r][0];
    for (int i = 1; i < NT / 32; ++i) mx = fmaxf(mx, s_w1[r][i]);
    float sum = 0.f;
    for (int i = 0; i < NT / 32; ++i) sum += s_we[r][i] * (s_w1[r][i] == mx ? 1.f : expf(s_w1[r][i] - mx));
    s_mx[r] = mx; s_den[r] = log_domain ? logf(sum) : sum;
  }
  __syncthreads();
  // ---- fast path: any L actual candidates bound the L-th best candidate from below.  tau = the L-th largest score
  // among the two largest logits of every (row, warp) -- 16 per row.  (With only the two largest per ROW the bound is
  // loose whenever the best L candidates come from one beam: additive probability scores make that the common case
  // for a flat distribution, thousands of candidates passed and the slow path below ran: +1.8 ms per beam-5 decode.)
  // Only candidates with score >= tau (about L of them) have to be collected and ranked.
  {
    if (threadIdx.x < 32) {
      constexpr int PER = 2 * (NT / 32);               // bound candidates per row
      const int lane = threadIdx.x, total = kin * PER;
      float cs[(KMAX * PER + 31) / 32];
#pragma unroll
      for (int u = 0; u < (KMAX * PER + 31) / 32; ++u) {
        const int e = lane + 32 * u;
        float sc = -INFINITY;
        if (e < total) {
          const int r = e / PER, w = (e % PER) >> 1;
          const float lg = (e & 1) ? s_w2[r][w] : s_w1[r][w];
          if (lg > -INFINITY) {
            const float pv = prev ? prev[b * kin + r] : 0.f;
            sc = (log_domain ? (lg - s_mx[r] - s_den[r]) : (expf(lg - s_mx[r]) / s_den[r])) + pv;
          }
          if constexpr (EOS) {                         // a finished row's single candidate
            if (s_fin[r] && e % PER == 0) sc = prev ? prev[b * kin + r] : 0.f;
          }
        }
        cs[u] = sc;
      }
      float kth = -INFINITY;
      for (int round = 0; round < L; ++round) {        // L rounds of "largest remaining"
        float bs = -INFINITY;
        int bu = 0;
#pragma unroll
        for (int u = 0; u < (KMAX * PER + 31) / 32; ++u) if (cs[u] > bs) { bs = cs[u]; bu = u; }
        float ws = bs;
        int wl = lane;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float os = __shfl_xor_sync(0xffffffffu, ws, o);
          const int ol = __shfl_xor_sync(0xffffffffu, wl, o);
          if (os > ws || (os == ws && ol < wl)) { ws = os; wl = ol; }
        }
        kth = ws;
        if (lane == wl) {
#pragma unroll
          for (int u = 0; u < (KMAX * PER + 31) / 32; ++u) if (u == bu) cs[u] = -INFINITY;
        }
      }
      if (lane == 0) s_tau = kth;                      // -inf (fewer than L real candidates): everything passes
    }
    __syncthreads();
    const float tau = s_tau;
    for (int r = 0; r < kin; ++r) {
      if constexpr (EOS) {
        if (s_fin[r]) {
          const float pv = prev ? prev[b * kin + r] : 0.f;
          if (threadIdx.x == 0 && pv >= tau) {
            const int pos = atomicAdd(&c_n, 1);
            if (pos < CAND_CAP) { c_s[pos] = pv; c_i[pos] = r * V + eos.pad_idx; }
          }
          continue;
        }
      }
      const T* x = logits + ((int64_t)b * kin + r) * ldl;
      const float mx = s_mx[r], den = s_den[r], pv = prev ? prev[b * kin + r] : 0.f;
      float tl;                                        // logit whose score is tau, minus a safety margin
      if (log_domain) tl = tau - pv + mx + den;
      else { const float need = tau - pv; tl = need > 0.f ? mx + logf(need * den) : -INFINITY; }
      tl -= 1e-3f;
      for (int j0 = threadIdx.x * 8; j0 < V; j0 += NT * 8) {
        float v[8];
        const int n = load_chunk8(x, j0, V, vec, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (i >= n) break;
          const float xv = v[i];
          if (!(xv > tl)) continue;
          const float sc = (log_domain ? (xv - mx - den) : (expf(xv - mx) / den)) + pv;
          if (sc >= tau) {
            const int pos = atomicAdd(&c_n, 1);
            if (pos < CAND_CAP) { c_s[pos] = sc; c_i[pos] = r * V + j0 + i; }
          }
        }
      }
    }
    __syncthreads();
    const int cn = c_n;
    if (cn <= CAND_CAP) {
      if (threadIdx.x < 32) {                          // warp 0: L rounds of "best remaining candidate"
        const int lane = threadIdx.x;
        float kth = 0.f;
        for (int round = 0; round < L; ++round) {
          float bs = -INFINITY;
          int bi = 0x7fffffff, bp = -1;
          for (int e = lane; e < cn; e += 32)
            if (better(c_s[e], c_i[e], bs, bi)) { bs = c_s[e]; bi = c_i[e]; bp = e; }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const float os = __shfl_xor_sync(0xffffffffu, bs, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o), op = __shfl_xor_sync(0xffffffffu, bp, o);
            if (better(os, oi, bs, bi)) { bs = os; bi = oi; bp = op; }
          }
          if (lane == 0) {
            if (bp >= 0) { c_s[bp] = -INFINITY; c_i[bp] = 0x7fffffff; }
            if (round < kout) {
              out_score[b * kout + round] = bs;
              out_parent[b * kout + round] = bi / V;
              out_token[b * kout + round] = bi % V;
              kth = bs;
            } else if (gap) {
              gap[b] = kth - bs;
            }
          }
          __syncwarp();
        }
      }
      return;
    }
    // more than CAND_CAP candidates tie with tau (degenerate logits): exact but slow path below
  }
  beam_select_exact<T, EOS>(b, kin, V, logits, ldl, prev, kout, out_score, out_parent, out_token, gap, log_domain, s_mx,
                            s_den, h_s, h_i, h_t, EOS ? s_fin : nullptr, eos.pad_idx);
}

// The same selection fed with the classifier GEMM's ICAP_EPI_ROWSTATS buffer: (largest, second largest, sum exp(x -
// largest)) per row and 128 logits.  No pass over the logits at all: the row statistics and the candidate bound come from
// the V / 128 partials per row, and only the ~L segments whose maximum can beat the bound are read.  Built for latency
// (the kernel sits on the decode step's critical path between the classifier and the next step's embedding): all rows'
// partials are requested at once, the bound and the final order are rank counts instead of L rounds of warp reductions.
constexpr int HIT_CAP = 256;

// (largest, second largest, sum exp(x - largest)) of two disjoint sets -> of their union
__device__ __forceinline__ void top2sum_merge(float& t1, float& t2, float& es, float o1, float o2, float oe) {
  const float n1 = fmaxf(t1, o1);
  // a side whose maximum IS the new maximum keeps its sum as it is (also keeps -inf - -inf out of the exponent)
  const float a = t1 == n1 ? 1.f : __expf(t1 - n1), c = o1 == n1 ? 1.f : __expf(o1 - n1);
  es = es * a + oe * c;
  t2 = fmaxf(fminf(t1, o1), fmaxf(t2, o2));
  t1 = n1;
}

template <typename T, bool EOS = false>
__global__ void __launch_bounds__(NT)
beam_select_stats_kernel(int kin, int V, const T* __restrict__ logits, int64_t ldl, const float* __restrict__ prev,
                         int kout, float* __restrict__ out_score, int* __restrict__ out_parent,
                         int* __restrict__ out_token, float* __restrict__ gap, int log_domain,
                         const float* __restrict__ stats, int64_t stats_ld, EosArgs eos) {
  pdl_prologue();
  constexpr int NW = NT / 32, PER = 2 * NW;
  __shared__ float s_mx[KMAX], s_den[KMAX], s_pv[KMAX], s_tl[KMAX];
  __shared__ float s_w1[KMAX][NW], s_w2[KMAX][NW];     // two largest logits of every (row, lane group)
  __shared__ float b_s[KMAX * PER];
  __shared__ float s_tau;
  __shared__ int h_n, c_n;
  __shared__ int h_seg[HIT_CAP];
  __shared__ float c_s[CAND_CAP];
  __shared__ int c_i[CAND_CAP];
  __shared__ float r_s[KMAX + 1];
  __shared__ float h_s[NT];
  __shared__ int h_i[NT], h_t[NT];
  __shared__ int s_fin[KMAX];                          // EOS: row r is finished
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = kout + 1, np = (V + 127) / 128;
  const float4* sp0 = reinterpret_cast<const float4*>(stats + (int64_t)b * kin * stats_ld);
  const int64_t sld4 = stats_ld >> 2;
  static_assert(KMAX <= NW, "one warp per beam row");
  if (tid == 0) { h_n = 0; c_n = 0; }
  if (tid <= KMAX) r_s[tid] = -INFINITY;
  // ---- warp r owns row r: softmax maximum / sum of the row and, as candidates for the bound, the two largest logits of each
  // of 8 lane groups (partials pi with pi % 32 in [4g, 4g + 4)).  A loop and five shuffle rounds: small code -- the first
  // version, unrolled over the rows, spent 40 % of its samples waiting for instruction fetches.
  bool fin = false;                                    // EOS: a finished row reads no statistics, offers one candidate
  if constexpr (EOS) {
    if (warp < kin) {
      fin = eos_finished(eos, b * kin + warp);
      if (lane == 0) s_fin[warp] = fin;
      if (fin) {
        if (lane < NW) { s_w1[warp][lane] = -INFINITY; s_w2[warp][lane] = -INFINITY; }
        if (lane == 0) { s_mx[warp] = 0.f; s_den[warp] = 0.f; s_pv[warp] = prev ? prev[b * kin + warp] : 0.f; }
      }
    }
  }
  if (warp < kin && !fin) {
    const int r = warp;
    const float4* sp = sp0 + r * sld4;
    float t1 = -INFINITY, t2 = -INFINITY, es = 0.f;
#pragma unroll 2
    for (int pi = lane; pi < np; pi += 32) {
      const float4 q = __ldg(sp + pi);
      top2sum_merge(t1, t2, es, q.x, q.y, q.z);
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      if (o == 4 && (lane & 3) == 0) { s_w1[r][lane >> 2] = t1; s_w2[r][lane >> 2] = t2; }
      const float o1 = __shfl_xor_sync(0xffffffffu, t1, o), o2 = __shfl_xor_sync(0xffffffffu, t2, o);
      const float oe = __shfl_xor_sync(0xffffffffu, es, o);
      top2sum_merge(t1, t2, es, o1, o2, oe);
    }
    if (lane == 0) {
      s_mx[r] = t1; s_den[r] = log_domain ? logf(es) : es;
      s_pv[r] = prev ? prev[b * kin + r] : 0.f;
    }
  }
  __syncthreads();
  // ---- bound: the L-th largest score among the two largest logits of every (row, warp) -- real candidates, so at least L
  // candidates reach it.  One rank count per bound candidate instead of L rounds of warp reductions.
  const int total = kin * PER;
  if (tid < total) {
    const int r = tid / PER, w = (tid % PER) >> 1;
    const float lg = (tid & 1) ? s_w2[r][w] : s_w1[r][w];
    float sc = -INFINITY;
    if (lg > -INFINITY) sc = (log_domain ? (lg - s_mx[r] - s_den[r]) : (__expf(lg - s_mx[r]) / s_den[r])) + s_pv[r];
    if constexpr (EOS) {
      if (s_fin[r] && tid % PER == 0) sc = s_pv[r];
    }
    b_s[tid] = sc;
  }
  __syncthreads();
  if (tid < total) {
    const float sc = b_s[tid];
    int rank = 0;
#pragma unroll 4
    for (int f = 0; f < total; ++f) {
      const float o = b_s[f];
      rank += (o > sc || (o == sc && f < tid)) ? 1 : 0;
    }
    if (rank == L - 1) s_tau = sc;                     // -inf (fewer than L real candidates): everything passes
  }
  __syncthreads();
  const float tau = s_tau;
  if (tid < kin) {                                     // logit whose score is tau, minus a safety margin
    const int r = tid;
    float tl;
    if (log_domain) tl = tau - s_pv[r] + s_mx[r] + s_den[r];
    else { const float need = tau - s_pv[r]; tl = need > 0.f ? s_mx[r] + logf(need * s_den[r]) : -INFINITY; }
    s_tl[r] = tl - 1e-3f;
  }
  __syncthreads();
  // ---- the 128-logit segments whose maximum exceeds tl (about L of kin * V / 128) ...
  if constexpr (EOS) {
    if (fin && lane == 0 && s_pv[warp] >= tau) {
      const int pos = atomicAdd(&c_n, 1);
      if (pos < CAND_CAP) { c_s[pos] = s_pv[warp]; c_i[pos] = warp * V + eos.pad_idx; }
    }
  }
  if (warp < kin && !fin) {
    const int r = warp;
    const float tl = s_tl[r];
    const float4* sp = sp0 + r * sld4;
#pragma unroll 2
    for (int pi = lane; pi < np; pi += 32) {
      if (__ldg(&sp[pi].x) > tl) {                     // L1 hit: read a moment ago
        const int pos = atomicAdd(&h_n, 1);
        if (pos < HIT_CAP) h_seg[pos] = (r << 20) | pi;
      }
    }
  }
  __syncthreads();
  // ---- ... are read, one warp per segment, and their candidates (score >= tau) collected
  const int nh = h_n;
  if (nh <= HIT_CAP) {
#pragma unroll 1
    for (int h = warp; h < nh; h += NW) {
      const int r = h_seg[h] >> 20, seg = h_seg[h] & 0xfffff;
      const T* x = logits + ((int64_t)b * kin + r) * ldl;
      const float mx = s_mx[r], den = s_den[r], pv = s_pv[r], tl = s_tl[r];
      const int j0 = seg * 128 + lane * 4;
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = j0 + i < V ? to_f32(x[j0 + i]) : -INFINITY;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (!(v[i] > tl)) continue;
        const float sc = (log_domain ? (v[i] - mx - den) : (__expf(v[i] - mx) / den)) + pv;
        if (sc >= tau) {
          const int pos = atomicAdd(&c_n, 1);
          if (pos < CAND_CAP) { c_s[pos] = sc; c_i[pos] = r * V + j0 + i; }
        }
      }
    }
  }
  __syncthreads();
  const int cn = c_n;
  if (nh <= HIT_CAP && cn <= CAND_CAP) {
    // ---- final order: every candidate counts the candidates that beat it
#pragma unroll 1
    for (int e = tid; e < cn; e += NT) {
      const float sc = c_s[e];
      const int ci = c_i[e];
      int rank = 0;
#pragma unroll 4
      for (int f = 0; f < cn; ++f) rank += better(c_s[f], c_i[f], sc, ci) ? 1 : 0;
      if (rank < L) {
        r_s[rank] = sc;
        if (rank < kout) {
          out_score[b * kout + rank] = sc;
          out_parent[b * kout + rank] = ci / V;
          out_token[b * kout + rank] = ci % V;
        }
      }
    }
    if (gap) {
      __syncthreads();
      if (tid == 0) gap[b] = r_s[kout - 1] - r_s[kout];
    }
    return;
  }
  // too many segments / candidates tie with the bound (degenerate logits): exact path over the logits
  beam_select_exact<T, EOS>(b, kin, V, logits, ldl, prev, kout, out_score, out_parent, out_token, gap, log_domain, s_mx,
                            s_den, h_s, h_i, h_t, EOS ? s_fin : nullptr, eos.pad_idx);
}

// ------------------------------------------------------------------------------------------------------------------
// PolicyNetwork.sample (model_RL.py:93-97): log_probs = log_softmax(output, dim=2); sequence = argmax(log_probs, dim=2).
// One block per (b, t) row of the fp32 logits: max + first arg-max, sum of exponentials, then the log-probabilities.
// The backward of the log-softmax (the self-critical loss back-propagates through the gathered log-probabilities,
// loss.py:90-103,145-158):  dx = dlogp - exp(logp) * sum_j dlogp_j.
__global__ void __launch_bounds__(NT)
log_softmax_argmax_kernel(int V, const float* __restrict__ x, int64_t ldx, float* __restrict__ logp, int64_t ldo,
                          long long* __restrict__ idx) {
  pdl_prologue();
  __shared__ float red[NT / 32];
  __shared__ float sv[NT];
  __shared__ int si[NT];
  const float* xr = x + (int64_t)blockIdx.x * ldx;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int j = threadIdx.x; j < V; j += NT) {
    const float v = xr[j];
    if (v > best) { best = v; bi = j; }            // ascending j per thread: the first maximum is kept
  }
  sv[threadIdx.x] = best; si[threadIdx.x] = bi;
  __syncthreads();
  for (int s = NT / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      const float b = sv[threadIdx.x + s];
      const int ib = si[threadIdx.x + s];
      if (b > sv[threadIdx.x] || (b == sv[threadIdx.x] && ib < si[threadIdx.x])) { sv[threadIdx.x] = b; si[threadIdx.x] = ib; }
    }
    __syncthreads();
  }
  const float mx = sv[0];
  float sum = 0.f;
  for (int j = threadIdx.x; j < V; j += NT) sum += expf(xr[j] - mx);
  sum = block_sum(sum, red);
  const float lse = mx + logf(sum);
  float* out = logp + (int64_t)blockIdx.x * ldo;
  for (int j = threadIdx.x; j < V; j += NT) out[j] = xr[j] - lse;
  if (threadIdx.x == 0 && idx) idx[blockIdx.x] = si[0];
}

__global__ void __launch_bounds__(NT)
log_softmax_bwd_kernel(int V, const float* __restrict__ logp, int64_t ldp, const float* __restrict__ dlogp, int64_t ldd,
                       float* __restrict__ dx, int64_t ldx) {
  pdl_prologue();
  __shared__ float red[NT / 32];
  const float* g = dlogp + (int64_t)blockIdx.x * ldd;
  const float* lp = logp + (int64_t)blockIdx.x * ldp;
  float sum = 0.f;
  for (int j = threadIdx.x; j < V; j += NT) sum += g[j];
  sum = block_sum(sum, red);
  float* out = dx + (int64_t)blockIdx.x * ldx;
  for (int j = threadIdx.x; j < V; j += NT) out[j] = g[j] - expf(lp[j]) * sum;
}

// tokens_out[b, s, 0..t] = tokens_in[b, parent[b,s], 0..t]; tokens_out[b, s, t+1] = token[b,s]
// the same gather is applied to the KV-cache slot table (which physical row holds position t')
__global__ void beam_reorder_kernel(int B, int k, int Tmax, int t, const int* __restrict__ parent,
                                    const int* __restrict__ token, const int* __restrict__ tok_in,
                                    int* __restrict__ tok_out, const int* __restrict__ slot_in,
                                    int* __restrict__ slot_out) {
  pdl_prologue();
  const int row = blockIdx.x;            // b*k + s
  const int b = row / k;
  const int src = b * k + parent[row];
  for (int j = threadIdx.x; j <= t + 1 && j < Tmax; j += blockDim.x) {
    tok_out[(int64_t)row * Tmax + j] = (j == t + 1) ? token[row] : tok_in[(int64_t)src * Tmax + j];
    if (slot_in) slot_out[(int64_t)row * Tmax + j] = (j == t + 1) ? row : slot_in[(int64_t)src * Tmax + j];
  }
}

// End of an <END>-aware beam search, one warp per image: lane s measures hypothesis s (generated tokens up to and including
// the first end_idx; before a first pad_idx; Tmax - 1 if neither), normalises its score by ((5 + len) / 6)^alpha, and
// ranks it by a count over the k normalised scores (ties: lower beam index); the warp then copies the n best token rows.
__global__ void __launch_bounds__(32)
beam_finalize_kernel(int k, int Tmax, const int* __restrict__ tokens, const float* __restrict__ score, int end_idx,
                     int pad_idx, float alpha, int n, int* __restrict__ out_ids, float* __restrict__ out_score,
                     int* __restrict__ out_len) {
  pdl_prologue();
  const int b = blockIdx.x, lane = threadIdx.x;
  int len = 0;
  float sc = 0.f, nrm = -INFINITY;
  if (lane < k) {
    const int* row = tokens + ((int64_t)b * k + lane) * Tmax;
    len = Tmax - 1;
    for (int j = 1; j < Tmax; ++j) {
      const int tk = row[j];
      if (tk == end_idx) { len = j; break; }
      if (tk == pad_idx) { len = j - 1; break; }
    }
    sc = score[b * k + lane];
    nrm = sc / powf((5.f + (float)len) / 6.f, alpha);
  }
  int rank = 0;
  for (int s = 0; s < k; ++s) {
    const float o = __shfl_sync(0xffffffffu, nrm, s);
    rank += (o > nrm || (o == nrm && s < lane)) ? 1 : 0;
  }
  if (lane < k && rank < n) {
    out_score[b * n + rank] = sc;
    out_len[b * n + rank] = len;
  }
  for (int s = 0; s < k; ++s) {
    const int rs = __shfl_sync(0xffffffffu, rank, s);
    if (rs >= n) continue;
    const int* src = tokens + ((int64_t)b * k + s) * Tmax;
    int* dst = out_ids + ((int64_t)b * n + rs) * Tmax;
    for (int j = lane; j < Tmax; j += 32) dst[j] = src[j];
  }
}

template <bool EOS>
void launch_beam_select(int dtype, int64_t B, int64_t kin, int64_t V, const void* logits, int64_t ldl,
                        const float* prev_score, int64_t kout, float* out_score, int* out_parent, int* out_token, float* gap,
                        int log_domain, const float* stats, int64_t stats_ld, EosArgs eos, cudaStream_t st) {
  dispatch_act(dtype, [&](auto tag) {
    using T = decltype(tag);
    if (stats)
      icap_launch(beam_select_stats_kernel<T, EOS>, (unsigned)B, NT, 0, st, kin, V, logits, ldl, prev_score, kout, out_score,
                  out_parent, out_token, gap, log_domain, stats, stats_ld, eos);
    else
      icap_launch(beam_select_kernel<T, EOS>, (unsigned)B, NT, 0, st, kin, V, logits, ldl, prev_score, kout, out_score,
                  out_parent, out_token, gap, log_domain, eos);
  });
}

}  // namespace

extern "C" int icap_xent(int dtype, int64_t M, int64_t V, void* logits, int64_t ldl, const int* targets,
                         int ignore_index, const float* inv_count, float* row_loss, int write_grad, void* stream) {
  ICAP_ARG(M > 0 && V > 0 && logits && targets && row_loss && inv_count, "icap_xent: null/empty argument");
  ICAP_ARG(ldl >= V && V < (1ll << 31) && M < (1ll << 31), "icap_xent: bad logits shape");
  const int esz = dtype == ICAP_F32 ? 4 : 2;
  const int vec = ((uintptr_t)logits % 16 == 0) && ((ldl * esz) % 16 == 0);
  size_t smem = (size_t)V * 4;
  int cached = smem <= 200 * 1024;
  if (!cached) smem = 0;
  cudaStream_t st = (cudaStream_t)stream;
  static IcapEnv e_reg;
  if (dtype == ICAP_BF16 && vec && V % 8 == 0 && V <= 5 * NT * 8 && e_reg.geti("ICAP_XENT_REG", 1) != 0) {
    icap_launch(xent_reg_kernel<5>, (unsigned)M, NT, 0, st, (int)V, (bf16*)logits, ldl, targets, ignore_index, inv_count,
                row_loss, write_grad);
    ICAP_LAUNCH_CHECK("icap_xent");
    return 0;
  }
  const int rc = dispatch_act(dtype, [&](auto tag) {
    if (int rc = ensure_smem<xent_kernel<decltype(tag)>>(smem)) return rc;
    icap_launch(xent_kernel<decltype(tag)>, (unsigned)M, NT, smem, st, V, logits, ldl, targets, ignore_index, inv_count,
                row_loss, write_grad, cached, vec);
    return 0;
  });
  if (rc) return rc;
  ICAP_LAUNCH_CHECK("icap_xent");
  return 0;
}

extern "C" int icap_xent_finalize(int64_t M, const float* row_loss, const float* inv_count, int focal, float* out2,
                                  void* stream) {
  ICAP_ARG(M > 0 && row_loss && inv_count && out2, "icap_xent_finalize: null/empty argument");
  ICAP_ARG(M < (1ll << 31), "icap_xent_finalize: too many rows");
  icap_launch(xent_finalize_kernel, 1, NT, 0, (cudaStream_t)stream, (int)M, row_loss, inv_count, focal, out2);
  ICAP_LAUNCH_CHECK("icap_xent_finalize");
  return 0;
}

extern "C" int icap_argmax(int dtype, int64_t M, int64_t V, const void* logits, int64_t ldl, int* out,
                           int64_t out_stride, float* gap, void* stream) {
  ICAP_ARG(M > 0 && V > 0 && logits && out, "icap_argmax: null/empty argument");
  ICAP_ARG(ldl >= V && V < (1ll << 31) && M < (1ll << 31), "icap_argmax: bad logits shape");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(argmax_kernel<decltype(tag)>, (unsigned)M, NT, 0, st, V, logits, ldl, out, out_stride, gap);
  });
  ICAP_LAUNCH_CHECK("icap_argmax");
  return 0;
}

extern "C" int icap_sample_tokens(int dtype, int64_t M, int64_t V, const void* logits, int64_t ldl, float inv_temperature,
                                  uint64_t seed, const int* seed_dev, int64_t t, int64_t Tmax, int* tokens, float* logp,
                                  int64_t ldp, int end_idx, int pad_idx, void* stream) {
  ICAP_ARG(M > 0 && V > 0 && logits && tokens && logp, "icap_sample_tokens: null/empty argument");
  ICAP_ARG(isfinite(inv_temperature) && inv_temperature > 0.f,
           "icap_sample_tokens: the temperature must be finite and > 0 (inverse %g)", (double)inv_temperature);
  ICAP_ARG(ldl >= V && V < (1 << 30) && M < (1ll << 31), "icap_sample_tokens: bad logits shape");
  ICAP_ARG(t >= 0 && t + 1 < Tmax && ldp > t, "icap_sample_tokens: position %lld out of range", (long long)t);
  cudaStream_t st = (cudaStream_t)stream;
  dispatch_act(dtype, [&](auto tag) {
    icap_launch(sample_kernel<decltype(tag)>, (unsigned)M, NT, 0, st, V, logits, ldl, inv_temperature, seed, seed_dev, t, Tmax,
                tokens, logp, ldp, end_idx, pad_idx);
  });
  ICAP_LAUNCH_CHECK("icap_sample_tokens");
  return 0;
}

extern "C" int icap_beam_select(int dtype, int64_t B, int64_t kin, int64_t V, const void* logits, int64_t ldl,
                                const float* prev_score, int64_t kout, float* out_score, int* out_parent,
                                int* out_token, float* gap, int log_domain, const float* stats, int64_t stats_ld,
                                void* stream) {
  ICAP_ARG(stats == nullptr || (((uintptr_t)stats & 15) == 0 && stats_ld % 4 == 0 && stats_ld >= 4 * ((V + 127) / 128)),
           "icap_beam_select: the statistics buffer needs 16-byte alignment and >= 4 * ceil(V / 128) floats per row");
  ICAP_ARG(B > 0 && V > 0 && logits && out_score && out_parent && out_token, "icap_beam_select: null/empty argument");
  ICAP_ARG(kin >= 1 && kin <= KMAX && kout >= 1 && kout <= KMAX, "icap_beam_select: beam width must be in [1, %d]", KMAX);
  ICAP_ARG(kin * V > kout, "icap_beam_select: fewer candidates than beams");
  ICAP_ARG(stats == nullptr || V < (1 << 27), "icap_beam_select: V too large for the statistics path");
  launch_beam_select<false>(dtype, B, kin, V, logits, ldl, prev_score, kout, out_score, out_parent, out_token, gap,
                            log_domain, stats, stats_ld, EosArgs{}, (cudaStream_t)stream);
  ICAP_LAUNCH_CHECK("icap_beam_select");
  return 0;
}

extern "C" int icap_beam_select_eos(int dtype, int64_t B, int64_t kin, int64_t V, const void* logits, int64_t ldl,
                                    const float* prev_score, int64_t kout, float* out_score, int* out_parent,
                                    int* out_token, float* gap, int log_domain, const float* stats, int64_t stats_ld,
                                    const int* tokens, int64_t Tmax, int64_t t, int end_idx, int pad_idx, void* stream) {
  ICAP_ARG(stats == nullptr || (((uintptr_t)stats & 15) == 0 && stats_ld % 4 == 0 && stats_ld >= 4 * ((V + 127) / 128)),
           "icap_beam_select_eos: the statistics buffer needs 16-byte alignment and >= 4 * ceil(V / 128) floats per row");
  ICAP_ARG(B > 0 && V > 0 && logits && out_score && out_parent && out_token && tokens,
           "icap_beam_select_eos: null/empty argument");
  ICAP_ARG(kin >= 1 && kin <= KMAX && kout >= 1 && kout <= KMAX, "icap_beam_select_eos: beam width must be in [1, %d]",
           KMAX);
  ICAP_ARG(log_domain == 1, "icap_beam_select_eos: scores are log-probabilities (log_domain = 1)");
  ICAP_ARG(t >= 0 && t + 1 < Tmax && Tmax < (1 << 30), "icap_beam_select_eos: position %lld out of range", (long long)t);
  ICAP_ARG(pad_idx >= 0 && pad_idx < V, "icap_beam_select_eos: pad_idx must be a token");
  // at t >= 1 every row offers at least one candidate (a finished row exactly one); at t = 0 no row is finished
  ICAP_ARG(t >= 1 ? kin >= kout : kin * V > kout, "icap_beam_select_eos: fewer candidates than beams");
  ICAP_ARG(stats == nullptr || V < (1 << 27), "icap_beam_select_eos: V too large for the statistics path");
  launch_beam_select<true>(dtype, B, kin, V, logits, ldl, prev_score, kout, out_score, out_parent, out_token, gap,
                           log_domain, stats, stats_ld, EosArgs{tokens, (int)Tmax, (int)t, end_idx, pad_idx},
                           (cudaStream_t)stream);
  ICAP_LAUNCH_CHECK("icap_beam_select_eos");
  return 0;
}

extern "C" int icap_beam_finalize(int64_t B, int64_t k, int64_t Tmax, const int* tokens, const float* score, int end_idx,
                                  int pad_idx, float alpha, int64_t n, int* out_ids, float* out_score, int* out_len,
                                  void* stream) {
  ICAP_ARG(B > 0 && Tmax > 1 && Tmax < (1 << 30) && tokens && score && out_ids && out_score && out_len,
           "icap_beam_finalize: null/empty argument");
  ICAP_ARG(k >= 1 && k <= KMAX && n >= 1 && n <= k, "icap_beam_finalize: need 1 <= n <= k <= %d", KMAX);
  ICAP_ARG(isfinite(alpha) && alpha >= 0.f, "icap_beam_finalize: the length penalty must be finite and >= 0 (%g)",
           (double)alpha);
  icap_launch(beam_finalize_kernel, (unsigned)B, 32, 0, (cudaStream_t)stream, (int)k, (int)Tmax, tokens, score, end_idx,
              pad_idx, alpha, (int)n, out_ids, out_score, out_len);
  ICAP_LAUNCH_CHECK("icap_beam_finalize");
  return 0;
}

extern "C" int icap_log_softmax_argmax(int64_t M, int64_t V, const float* x, int64_t ldx, float* logp, int64_t ldo,
                                       long long* idx, void* stream) {
  ICAP_ARG(M > 0 && V > 0 && x && logp, "icap_log_softmax_argmax: null/empty argument");
  ICAP_ARG(ldx >= V && ldo >= V && V < (1ll << 31) && M < (1ll << 31), "icap_log_softmax_argmax: bad logits shape");
  icap_launch(log_softmax_argmax_kernel, (unsigned)M, NT, 0, (cudaStream_t)stream, (int)V, x, ldx, logp, ldo, idx);
  ICAP_LAUNCH_CHECK("icap_log_softmax_argmax");
  return 0;
}

extern "C" int icap_log_softmax_bwd(int64_t M, int64_t V, const float* logp, int64_t ldp, const float* dlogp, int64_t ldd,
                                    float* dx, int64_t ldx, void* stream) {
  ICAP_ARG(M > 0 && V > 0 && logp && dlogp && dx, "icap_log_softmax_bwd: null/empty argument");
  ICAP_ARG(ldp >= V && ldd >= V && ldx >= V && V < (1ll << 31) && M < (1ll << 31),
           "icap_log_softmax_bwd: bad logits shape");
  icap_launch(log_softmax_bwd_kernel, (unsigned)M, NT, 0, (cudaStream_t)stream, (int)V, logp, ldp, dlogp, ldd, dx, ldx);
  ICAP_LAUNCH_CHECK("icap_log_softmax_bwd");
  return 0;
}

extern "C" int icap_beam_reorder(int64_t B, int64_t k, int64_t Tmax, int64_t t, const int* parent, const int* token,
                                 const int* tok_in, int* tok_out, const int* slot_in, int* slot_out, void* stream) {
  ICAP_ARG(B > 0 && k > 0 && parent && token && tok_in && tok_out, "icap_beam_reorder: null/empty argument");
  ICAP_ARG(tok_in != tok_out && (slot_in == nullptr || slot_in != slot_out), "icap_beam_reorder: must be out of place");
  icap_launch(beam_reorder_kernel, (unsigned)(B * k), 32, 0, (cudaStream_t)stream, (int)B, (int)k, (int)Tmax, (int)t, parent,
                                                                         token, tok_in, tok_out, slot_in, slot_out);
  ICAP_LAUNCH_CHECK("icap_beam_reorder");
  return 0;
}
