// Caption metrics on token ids: BLEU-1..4, ROUGE-L, CIDEr and CIDEr-D (coco-caption's bleu_scorer.py / rouge.py,
// pyciderevalcap's cider_scorer.py / ciderD_scorer.py), for evaluation (core/evaluations.py:12-34) and as the
// self-critical reward (loss.py:160-186).
//
// A row is read the way core/utils.py::decode_captions reads it: a <START> (1) at position 0 is skipped, <NULL> (0) is
// dropped, the row ends at the first <END> (2), which counts as a token ('.').  An n-gram (n = 1..4) of 15-bit ids packs
// into one uint64 without collisions:  n << 60 | t0 << 45 | t1 << 30 | t2 << 15 | t3  (missing positions 0).  Sorting
// the keys therefore groups them by order.
//
// Work split: one warp per row (cook, prep) / per image (df) / per candidate (score).  Everything is deterministic:
// fixed-order warp reductions in fp64, integer atomics only (document frequencies, corpus BLEU counts).
#include "icap_common.cuh"

namespace {

constexpr int kMaxWidth = 128;             // row width limit (MAX_LENGTH = 49 needs 52); 2 x 64-bit LCS words
constexpr int kStart = 1, kEnd = 2;
constexpr uint64_t kNoKey = ~0ull;         // sorts after every real key
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {       // splitmix64 finaliser
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}

__device__ __forceinline__ int key_order(uint64_t k) { return (int)(k >> 60); }

__device__ __forceinline__ int ngram_count(int len, int n) { return len - n + 1 > 0 ? len - n + 1 : 0; }

__device__ int table_df(const uint64_t* tk, const int* tdf, uint64_t mask, uint64_t key) {
  for (uint64_t h = mix64(key) & mask;; h = (h + 1) & mask) {
    const uint64_t k = tk[h];
    if (k == key) return tdf[h];
    if (k == 0) return 0;
  }
}

// first index of `key` in the sorted keys[0..n), or -1
__device__ __forceinline__ int find_key(const uint64_t* keys, int n, uint64_t key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (keys[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo < n && keys[lo] == key ? lo : -1;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

__host__ __device__ __forceinline__ int pow2_at_least(int n) {
  int p = 32;
  while (p < n) p <<= 1;
  return p;
}

// One warp cooks one row: toks[0..len) = the tokens after the cut, s[0..nk) = its distinct n-gram keys (ascending),
// cnt[0..nk) = their counts.  s / cnt hold pow2_at_least(4 * W) entries.  Returns nk; *len_out = len.
template <typename T>
__device__ int cook_row(const T* row, int W, uint64_t* s, int* cnt, int* toks, int lane, int* len_out) {
  const unsigned lt = (1u << lane) - 1u;
  int len = 0;
  for (int base = 0; base < W; base += 32) {
    const int p = base + lane;
    const int t = p < W ? (int)row[p] : 0;
    const unsigned endm = __ballot_sync(kFull, p < W && t == kEnd);
    const int first_end = endm ? __ffs(endm) - 1 : 32;
    const bool keep = p < W && lane <= first_end && t != 0 && !(p == 0 && t == kStart);
    const unsigned km = __ballot_sync(kFull, keep);
    if (keep) toks[len + __popc(km & lt)] = t;
    len += __popc(km);
    if (endm) break;
  }
  __syncwarp();
  int nvalid = 0, off[4];
#pragma unroll
  for (int n = 1; n <= 4; ++n) { off[n - 1] = nvalid; nvalid += ngram_count(len, n); }
  const int P = pow2_at_least(nvalid);
  for (int i = lane; i < P; i += 32) {
    uint64_t key = kNoKey;
    if (i < nvalid) {
      const int n = i >= off[3] ? 4 : i >= off[2] ? 3 : i >= off[1] ? 2 : 1;
      const int j = i - off[n - 1];
      key = (uint64_t)n << 60;
      for (int m = 0; m < n; ++m) key |= (uint64_t)toks[j + m] << (45 - 15 * m);
    }
    s[i] = key;
  }
  __syncwarp();
  for (int k = 2; k <= P; k <<= 1) {                 // bitonic sort of s[0..P)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < P; i += 32) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const uint64_t a = s[i], b = s[ixj];
          if ((a > b) == ((i & k) == 0)) { s[i] = b; s[ixj] = a; }
        }
      }
      __syncwarp();
    }
  }
  // compact run heads in place: head rank j <- key, cnt[j] <- run start, then cnt[j] = start[j+1] - start[j]
  int nk = 0;
  for (int base = 0; base < nvalid; base += 32) {
    const int i = base + lane;
    const uint64_t key = i < nvalid ? s[i] : kNoKey;
    const bool head = i < nvalid && (i == 0 || s[i - 1] != key);
    const unsigned hm = __ballot_sync(kFull, head);
    __syncwarp();
    if (head) { s[nk + __popc(hm & lt)] = key; cnt[nk + __popc(hm & lt)] = i; }
    nk += __popc(hm);
    __syncwarp();
  }
  for (int base = 0; base < nk; base += 32) {
    const int j = base + lane;
    const int c = j < nk ? (j + 1 < nk ? cnt[j + 1] : nvalid) - cnt[j] : 0;
    __syncwarp();
    if (j < nk) cnt[j] = c;
    __syncwarp();
  }
  *len_out = len;
  return nk;
}

// shared memory of one warp, a multiple of 16 bytes so that every warp's uint64 / double arrays stay aligned
__host__ __device__ __forceinline__ size_t cook_smem_bytes(int W) {
  const size_t b = (size_t)pow2_at_least(4 * W) * (sizeof(uint64_t) + sizeof(int)) + (size_t)W * sizeof(int);
  return (b + 15) & ~(size_t)15;
}

template <typename T>
__global__ void cook_kernel(const T* __restrict__ tokens, int N, int W, int64_t ld, uint64_t* __restrict__ keys,
                            int* __restrict__ counts, int* __restrict__ nkeys, int* __restrict__ lens,
                            int* __restrict__ toks_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  pdl_prologue();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= N) return;
  const int P = pow2_at_least(4 * W);
  unsigned char* mine = smem + (size_t)warp * cook_smem_bytes(W);
  uint64_t* s = reinterpret_cast<uint64_t*>(mine);
  int* cnt = reinterpret_cast<int*>(s + P);
  int* toks = cnt + P;
  int len;
  const int nk = cook_row(tokens + (int64_t)row * ld, W, s, cnt, toks, lane, &len);
  const int KW = 4 * W;
  for (int j = lane; j < KW; j += 32) {
    keys[(int64_t)row * KW + j] = j < nk ? s[j] : 0;
    counts[(int64_t)row * KW + j] = j < nk ? cnt[j] : 0;
  }
  for (int j = lane; j < W; j += 32) toks_out[(int64_t)row * W + j] = j < len ? toks[j] : 0;
  if (lane == 0) { nkeys[row] = nk; lens[row] = len; }
}

// One warp per image: every key of every ref is counted once per image (skipped when an earlier ref of the image
// holds it).  n_unique (nullable) += the number of such keys; table_keys != NULL: df[key] += 1.
__global__ void df_kernel(int n_img, const int64_t* __restrict__ img_off, int W, const uint64_t* __restrict__ keys,
                          const int* __restrict__ nkeys, unsigned long long* table_keys, int* table_df, uint64_t mask,
                          unsigned long long* n_unique) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int img = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (img >= n_img) return;
  const int64_t r0 = img_off[img], r1 = img_off[img + 1];
  const int KW = 4 * W;
  int counted = 0;
  for (int64_t r = r0; r < r1; ++r) {
    const uint64_t* kr = keys + r * KW;
    const int nk = nkeys[r];
    for (int j = lane; j < nk; j += 32) {
      const uint64_t key = kr[j];
      bool seen = false;
      for (int64_t q = r0; q < r && !seen; ++q) seen = find_key(keys + q * KW, nkeys[q], key) >= 0;
      if (seen) continue;
      ++counted;
      if (table_keys) {
        for (uint64_t h = mix64(key) & mask;; h = (h + 1) & mask) {
          const unsigned long long prev = atomicCAS(&table_keys[h], 0ull, (unsigned long long)key);
          if (prev == 0ull || prev == key) { atomicAdd(&table_df[h], 1); break; }
        }
      }
    }
  }
  counted = warp_sum_i(counted);
  if (n_unique && lane == 0 && counted) atomicAdd(n_unique, (unsigned long long)counted);
}

// One warp per ref: norms[r][n-1] = || count(g) * (log(n_img) - log(max(1, df(g)))) ||_2 over the n-grams of order n.
__global__ void ref_prep_kernel(int N, int W, const uint64_t* __restrict__ keys, const int* __restrict__ counts,
                                const int* __restrict__ nkeys, double ref_len, const uint64_t* __restrict__ tk,
                                const int* __restrict__ tdf, uint64_t mask, double* __restrict__ norms) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= N) return;
  const int KW = 4 * W, nk = nkeys[r];
  double acc[4] = {0, 0, 0, 0};
  for (int j = lane; j < nk; j += 32) {
    const uint64_t key = keys[(int64_t)r * KW + j];
    const int df = table_df(tk, tdf, mask, key);
    const double v = counts[(int64_t)r * KW + j] * (ref_len - log((double)max(1, df)));
    const int o = key_order(key) - 1;
#pragma unroll
    for (int n = 0; n < 4; ++n) if (n == o) acc[n] += v * v;
  }
#pragma unroll
  for (int n = 0; n < 4; ++n) {
    const double t = warp_sum_d(acc[n]);
    if (lane == 0) norms[(int64_t)r * 4 + n] = sqrt(t);
  }
}

__host__ __device__ __forceinline__ size_t score_smem_bytes(int Wc) {
  const size_t b = (size_t)pow2_at_least(4 * Wc) * (sizeof(uint64_t) + sizeof(double) + 2 * sizeof(int)) +
                   (size_t)Wc * sizeof(int);
  return (b + 15) & ~(size_t)15;
}

// One warp per candidate.  scores[m] = {CIDEr-D, CIDEr, ROUGE-L, BLEU-1..4} (nullable), reward[m] =
// cider_w * CIDEr-D + bleu_w * BLEU-4 (nullable), corpus (nullable) += {correct[4], guess[4], testlen, reflen}.
template <typename T>
__global__ void score_kernel(const T* __restrict__ cand, int M, int Wc, int64_t ldc, const int64_t* __restrict__ cand_img,
                             int n_img, const int64_t* __restrict__ img_off, int W, const uint64_t* __restrict__ keys,
                             const int* __restrict__ counts, const int* __restrict__ nkeys, const int* __restrict__ lens,
                             const int* __restrict__ rtoks, const double* __restrict__ norms,
                             const uint64_t* __restrict__ tk, const int* __restrict__ tdf, uint64_t mask,
                             float* __restrict__ scores, float* __restrict__ reward, float cider_w, float bleu_w,
                             unsigned long long* __restrict__ corpus) {
  extern __shared__ __align__(16) unsigned char smem[];
  pdl_prologue();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int m = blockIdx.x * (blockDim.x >> 5) + warp;
  if (m >= M) return;
  const int P = pow2_at_least(4 * Wc);
  unsigned char* mine = smem + (size_t)warp * score_smem_bytes(Wc);
  uint64_t* s = reinterpret_cast<uint64_t*>(mine);
  double* vc = reinterpret_cast<double*>(s + P);
  int* cnt = reinterpret_cast<int*>(vc + P);
  int* maxref = cnt + P;
  int* toks = maxref + P;
  int lc;
  const int nk = cook_row(cand + (int64_t)m * ldc, Wc, s, cnt, toks, lane, &lc);

  const double ref_len = log((double)n_img);
  const int64_t img = cand_img[m];
  const bool has_img = img >= 0 && img < n_img;
  const int64_t r0 = has_img ? img_off[img] : 0, r1 = has_img ? img_off[img + 1] : 0;

  // candidate vector: vc[k] = count * idf, norms per order
  double nc[4] = {0, 0, 0, 0};
  for (int k = lane; k < nk; k += 32) {
    const int df = table_df(tk, tdf, mask, s[k]);
    const double v = cnt[k] * (ref_len - log((double)max(1, df)));
    vc[k] = v;
    maxref[k] = 0;
    const int o = key_order(s[k]) - 1;
#pragma unroll
    for (int n = 0; n < 4; ++n) if (n == o) nc[n] += v * v;
  }
#pragma unroll
  for (int n = 0; n < 4; ++n) nc[n] = sqrt(warp_sum_d(nc[n]));
  __syncwarp();

  const int KW = 4 * W;
  const int len_c2 = ngram_count(lc, 2);
  double cider_d = 0.0, cider = 0.0, p_max = 0.0, r_max = 0.0;
  int reflen = -1;
  for (int64_t r = r0; r < r1; ++r) {
    const uint64_t* kr = keys + r * KW;
    const int* cr = counts + r * KW;
    const int nkr = nkeys[r], lr = lens[r];
    double dd[4] = {0, 0, 0, 0}, dc[4] = {0, 0, 0, 0};
    for (int k = lane; k < nk; k += 32) {
      const int j = find_key(kr, nkr, s[k]);
      if (j < 0) continue;
      const int c = cr[j];
      maxref[k] = max(maxref[k], c);
      const double idf = vc[k] / cnt[k];
      const double v_r = c * idf, v_c = vc[k];
      const int o = key_order(s[k]) - 1;
#pragma unroll
      for (int n = 0; n < 4; ++n) if (n == o) { dd[n] += fmin(v_c, v_r) * v_r; dc[n] += v_c * v_r; }
    }
    const double delta = (double)(len_c2 - ngram_count(lr, 2));
    const double pen = exp(-(delta * delta) / 72.0);          // 2 sigma^2, sigma = 6
    double sd = 0.0, sc = 0.0;
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      double a = warp_sum_d(dd[n]), b = warp_sum_d(dc[n]);
      const double nr = norms[r * 4 + n];
      if (nc[n] != 0.0 && nr != 0.0) { a /= nc[n] * nr; b /= nc[n] * nr; }
      sd += a * pen;
      sc += b;
    }
    cider_d += sd;
    cider += sc;
    // closest ref length, the shorter one on a tie
    if (reflen < 0 || abs(lr - lc) < abs(reflen - lc) || (abs(lr - lc) == abs(reflen - lc) && lr < reflen)) reflen = lr;
    // LCS (Allison-Dix bit vectors over the ref's positions, 128 bits)
    const int* rt = rtoks + r * W;
    int rv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) rv[q] = lane + 32 * q < lr ? rt[lane + 32 * q] : -1;
    uint64_t v0 = ~0ull, v1 = ~0ull;
    for (int i = 0; i < lc; ++i) {
      const int t = toks[i];
      const uint64_t m0 = (uint64_t)__ballot_sync(kFull, rv[0] == t) | (uint64_t)__ballot_sync(kFull, rv[1] == t) << 32;
      const uint64_t m1 = (uint64_t)__ballot_sync(kFull, rv[2] == t) | (uint64_t)__ballot_sync(kFull, rv[3] == t) << 32;
      const uint64_t u0 = v0 & m0, u1 = v1 & m1;
      const uint64_t s0 = v0 + u0;
      const uint64_t s1 = v1 + u1 + (s0 < v0 ? 1ull : 0ull);
      v0 = s0 | (v0 & ~m0);
      v1 = s1 | (v1 & ~m1);
    }
    const uint64_t live0 = lr >= 64 ? ~0ull : ((1ull << lr) - 1ull);
    const uint64_t live1 = lr >= 128 ? ~0ull : lr <= 64 ? 0ull : ((1ull << (lr - 64)) - 1ull);
    const int lcs = __popcll(~v0 & live0) + __popcll(~v1 & live1);
    if (lc > 0) p_max = fmax(p_max, (double)lcs / lc);
    if (lr > 0) r_max = fmax(r_max, (double)lcs / lr);
  }
  __syncwarp();
  const int nrefs = (int)(r1 - r0);
  if (nrefs > 0) {
    cider_d = 10.0 * (cider_d / 4.0) / nrefs;
    cider = 10.0 * (cider / 4.0) / nrefs;
  }
  if (reflen < 0) reflen = 0;

  int correct[4] = {0, 0, 0, 0};
  for (int k = lane; k < nk; k += 32) {
    const int c = min(cnt[k], maxref[k]);
    const int o = key_order(s[k]) - 1;
#pragma unroll
    for (int n = 0; n < 4; ++n) if (n == o) correct[n] += c;
  }
#pragma unroll
  for (int n = 0; n < 4; ++n) correct[n] = warp_sum_i(correct[n]);
  if (lane != 0) return;

  const double tiny = 1e-15, small = 1e-9;
  double bleu[4], prod = 1.0;
  const double ratio = (lc + tiny) / (reflen + small);
  const double bp = ratio < 1.0 ? exp(1.0 - 1.0 / ratio) : 1.0;
#pragma unroll
  for (int n = 0; n < 4; ++n) {
    prod *= (correct[n] + tiny) / (ngram_count(lc, n + 1) + small);
    bleu[n] = pow(prod, 1.0 / (n + 1)) * bp;
  }
  const double beta2 = 1.2 * 1.2;
  const double rouge = (p_max != 0.0 && r_max != 0.0) ? (1.0 + beta2) * p_max * r_max / (r_max + beta2 * p_max) : 0.0;
  if (scores) {
    float* o = scores + (int64_t)m * 7;
    o[0] = (float)cider_d; o[1] = (float)cider; o[2] = (float)rouge;
#pragma unroll
    for (int n = 0; n < 4; ++n) o[3 + n] = (float)bleu[n];
  }
  if (reward) reward[m] = (float)(cider_w * cider_d + bleu_w * bleu[3]);
  if (corpus) {
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      atomicAdd(&corpus[n], (unsigned long long)correct[n]);
      atomicAdd(&corpus[4 + n], (unsigned long long)ngram_count(lc, n + 1));
    }
    atomicAdd(&corpus[8], (unsigned long long)lc);
    atomicAdd(&corpus[9], (unsigned long long)reflen);
  }
}

int warps_per_block(size_t per_warp) {
  const size_t w = (48 * 1024) / per_warp;
  return (int)(w < 1 ? 1 : w > 4 ? 4 : w);
}

bool is_pow2(int64_t x) { return x > 0 && (x & (x - 1)) == 0; }

}  // namespace

extern "C" int icap_caption_cook(const void* tokens, int tok_is_int64, int64_t N, int64_t W, int64_t ld, uint64_t* keys,
                                 int* counts, int* nkeys, int* lens, int* toks, void* stream) {
  ICAP_ARG(N >= 0 && N < (1ll << 31), "icap_caption_cook: N=%lld out of range", (long long)N);
  ICAP_ARG(W >= 1 && W <= kMaxWidth, "icap_caption_cook: row width %lld outside [1, %d]", (long long)W, kMaxWidth);
  ICAP_ARG(ld >= W, "icap_caption_cook: ld=%lld < W=%lld", (long long)ld, (long long)W);
  if (N == 0) return 0;
  ICAP_ARG(tokens && keys && counts && nkeys && lens && toks, "icap_caption_cook: null pointer");
  const size_t per = cook_smem_bytes((int)W);
  const int wpb = warps_per_block(per);
  const dim3 grid((unsigned)ceil_div64(N, wpb)), block(32 * wpb);
  cudaStream_t st = (cudaStream_t)stream;
  if (tok_is_int64)
    icap_launch(cook_kernel<int64_t>, grid, block, per * wpb, st, (const int64_t*)tokens, (int)N, (int)W, ld, keys, counts,
                nkeys, lens, toks);
  else
    icap_launch(cook_kernel<int>, grid, block, per * wpb, st, (const int*)tokens, (int)N, (int)W, ld, keys, counts, nkeys,
                lens, toks);
  ICAP_LAUNCH_CHECK("icap_caption_cook");
  return 0;
}

extern "C" int icap_caption_df(int64_t n_img, const int64_t* img_off, int64_t W, const uint64_t* keys, const int* nkeys,
                               uint64_t* table_keys, int* table_df, int64_t cap, long long* n_unique, void* stream) {
  ICAP_ARG(n_img >= 1 && n_img < (1ll << 31), "icap_caption_df: n_img=%lld out of range", (long long)n_img);
  ICAP_ARG(W >= 1 && W <= kMaxWidth, "icap_caption_df: row width %lld outside [1, %d]", (long long)W, kMaxWidth);
  ICAP_ARG(img_off && keys && nkeys, "icap_caption_df: null pointer");
  ICAP_ARG(table_keys ? (table_df != nullptr && is_pow2(cap)) : n_unique != nullptr,
           "icap_caption_df: needs a table (power-of-two capacity, got %lld) or a counter", (long long)cap);
  const int wpb = 4;
  icap_launch(df_kernel, dim3((unsigned)ceil_div64(n_img, wpb)), dim3(32 * wpb), 0, (cudaStream_t)stream, (int)n_img,
              img_off, (int)W, keys, nkeys, (unsigned long long*)table_keys, table_df,
              (uint64_t)(table_keys ? cap - 1 : 0), (unsigned long long*)n_unique);
  ICAP_LAUNCH_CHECK("icap_caption_df");
  return 0;
}

extern "C" int icap_caption_ref_prep(int64_t N, int64_t W, const uint64_t* keys, const int* counts, const int* nkeys,
                                     int64_t n_img, const uint64_t* table_keys, const int* table_df, int64_t cap,
                                     double* norms, void* stream) {
  ICAP_ARG(N >= 1 && N < (1ll << 31) && n_img >= 1, "icap_caption_ref_prep: N=%lld / n_img=%lld out of range",
           (long long)N, (long long)n_img);
  ICAP_ARG(W >= 1 && W <= kMaxWidth, "icap_caption_ref_prep: row width %lld outside [1, %d]", (long long)W, kMaxWidth);
  ICAP_ARG(is_pow2(cap), "icap_caption_ref_prep: capacity %lld is not a power of two", (long long)cap);
  ICAP_ARG(keys && counts && nkeys && table_keys && table_df && norms, "icap_caption_ref_prep: null pointer");
  const int wpb = 4;
  icap_launch(ref_prep_kernel, dim3((unsigned)ceil_div64(N, wpb)), dim3(32 * wpb), 0, (cudaStream_t)stream, (int)N,
              (int)W, keys, counts, nkeys, log((double)n_img), table_keys, table_df, (uint64_t)(cap - 1), norms);
  ICAP_LAUNCH_CHECK("icap_caption_ref_prep");
  return 0;
}

extern "C" int icap_caption_score(const void* cand, int cand_is_int64, int64_t M, int64_t Wc, int64_t ldc,
                                  const int64_t* cand_img, int64_t n_img, const int64_t* img_off, int64_t W,
                                  const uint64_t* keys, const int* counts, const int* nkeys, const int* lens, const int* toks,
                                  const double* norms, const uint64_t* table_keys, const int* table_df, int64_t cap,
                                  float* scores, float* reward, float cider_weight, float bleu_weight, long long* corpus,
                                  void* stream) {
  ICAP_ARG(M >= 0 && M < (1ll << 31), "icap_caption_score: M=%lld out of range", (long long)M);
  ICAP_ARG(Wc >= 1 && Wc <= kMaxWidth, "icap_caption_score: candidate width %lld outside [1, %d]", (long long)Wc, kMaxWidth);
  ICAP_ARG(W >= 1 && W <= kMaxWidth, "icap_caption_score: reference width %lld outside [1, %d]", (long long)W, kMaxWidth);
  ICAP_ARG(ldc >= Wc, "icap_caption_score: ldc=%lld < Wc=%lld", (long long)ldc, (long long)Wc);
  ICAP_ARG(n_img >= 1 && n_img < (1ll << 31), "icap_caption_score: n_img=%lld out of range", (long long)n_img);
  ICAP_ARG(is_pow2(cap), "icap_caption_score: capacity %lld is not a power of two", (long long)cap);
  if (M == 0) return 0;
  ICAP_ARG(cand && cand_img && img_off && keys && counts && nkeys && lens && toks && norms && table_keys && table_df,
           "icap_caption_score: null pointer");
  const size_t per = score_smem_bytes((int)Wc);
  const int wpb = warps_per_block(per);
  const dim3 grid((unsigned)ceil_div64(M, wpb)), block(32 * wpb);
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t mask = (uint64_t)(cap - 1);
  if (cand_is_int64)
    icap_launch(score_kernel<int64_t>, grid, block, per * wpb, st, (const int64_t*)cand, (int)M, (int)Wc, ldc, cand_img,
                (int)n_img, img_off, (int)W, keys, counts, nkeys, lens, toks, norms, table_keys, table_df, mask, scores,
                reward, cider_weight, bleu_weight, (unsigned long long*)corpus);
  else
    icap_launch(score_kernel<int>, grid, block, per * wpb, st, (const int*)cand, (int)M, (int)Wc, ldc, cand_img, (int)n_img,
                img_off, (int)W, keys, counts, nkeys, lens, toks, norms, table_keys, table_df, mask, scores, reward,
                cider_weight, bleu_weight, (unsigned long long*)corpus);
  ICAP_LAUNCH_CHECK("icap_caption_score");
  return 0;
}
