// Graph scoring (gather-sum of rows of M in NumPy's pairwise order) and masked top-N.
//
// Replaces reference src/scripts/recommend.py:7-18 (simple_recs), cut_cards.py:7-18
// (simple_cuts) and the ranking walk of src/scripts/ml_recommend.py:87-104 /
// web/ml_recommend_web.py:46-60.
#include "cc_common.cuh"

namespace cc {

// ------------------------------------------------------------- pairwise gather
// recommend.py:10-13 sums an F-ordered fancy-index copy along its contiguous axis, so
// NumPy evaluates every column with its pairwise algorithm (blocks <= 128 rows with 8
// interleaved accumulators, recursive halving above that).  Reproducing that order
// makes the float64 scores bit-identical to the reference's, hence identical ranks.
struct Leaf { int32_t start, len, merges, cube; };

__global__ void __launch_bounds__(128)
gather_leaf_kernel(const double* __restrict__ m, int64_t ld, int32_t num_cards,
                   const int32_t* __restrict__ rows, const int64_t* __restrict__ row_ptr,
                   const Leaf* __restrict__ leaves, int zero_diag, double* __restrict__ partial) {
  const Leaf lf = leaves[blockIdx.y];
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= num_cards) return;
  const int32_t* r = rows + row_ptr[lf.cube] + lf.start;
  auto at = [&](int k) -> double {
    const int32_t i = r[k];
    return (zero_diag && i == j) ? 0.0 : m[int64_t(i) * ld + j];
  };
  double res;
  const int n = lf.len;
  if (n < 8) {
    res = 0.0;
    for (int k = 0; k < n; ++k) res += at(k);
  } else {
    double a[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) a[q] = at(q);
    int k = 8;
    for (; k < n - (n % 8); k += 8) {
#pragma unroll
      for (int q = 0; q < 8; ++q) a[q] += at(k + q);
    }
    res = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
    for (; k < n; ++k) res += at(k);
  }
  partial[int64_t(blockIdx.y) * num_cards + j] = res;
}

__global__ void __launch_bounds__(128)
gather_combine_kernel(const double* __restrict__ partial, int32_t num_cards, const Leaf* __restrict__ leaves,
                      const int32_t* __restrict__ leaf_ptr, double* __restrict__ scores, int64_t ld_scores) {
  const int cube = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= num_cards) return;
  double stack[24];
  int sp = 0;
  for (int l = leaf_ptr[cube]; l < leaf_ptr[cube + 1]; ++l) {
    stack[sp++] = partial[int64_t(l) * num_cards + j];
    for (int mgs = leaves[l].merges; mgs > 0; --mgs) {
      const double b = stack[--sp];
      stack[sp - 1] = stack[sp - 1] + b;
    }
  }
  // ufunc reduce starts from the additive identity: out = 0.0 + pairwise(...)
  scores[int64_t(cube) * ld_scores + j] = sp > 0 ? 0.0 + stack[0] : 0.0;
}

// ---------------------------------------------------------------- masked top-N
// (the composite key, KeyOf / make_key, and the raw-value bound rs_raw_bound live in cc_common.cuh: rank.cu
// ranks by the same order)
constexpr int TOPN_THREADS = 512;
constexpr int TOPN_MAX_SMEM_N = 2048;

template <typename T>
__global__ void __launch_bounds__(TOPN_THREADS)
topn_masked_kernel(const T* __restrict__ scores, int64_t ld, int32_t num_cards,
                   const int64_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_idx,
                   int mode_only_listed, int descending, int32_t n, int32_t n_pad,
                   int32_t* __restrict__ out_ids, T* __restrict__ out_vals, int32_t* __restrict__ out_count) {
  using KO = KeyOf<T>;
  using K = typename KO::K;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  K* cand = reinterpret_cast<K*>(smem_raw);                          // n_pad keys
  uint32_t* mask = reinterpret_cast<uint32_t*>(cand + n_pad);        // ceil(C/32) words
  __shared__ int hist[256];
  __shared__ int s_need, s_bucket, s_digit, s_cnt;

  const int cube = blockIdx.x;
  const T* sc = scores + int64_t(cube) * ld;
  const int words = (num_cards + 31) >> 5;
  for (int w = threadIdx.x; w < words; w += blockDim.x) mask[w] = 0;
  __syncthreads();
  const int64_t mb = mask_ptr[cube], me = mask_ptr[cube + 1];
  for (int64_t p = mb + threadIdx.x; p < me; p += blockDim.x) {
    const int32_t c = mask_idx[p];
    if (c >= 0 && c < num_cards) atomicOr(&mask[c >> 5], 1u << (c & 31));
  }
  __syncthreads();
  // number of candidates
  int local = 0;
  for (int w = threadIdx.x; w < words; w += blockDim.x) local += __popc(mask[w]);
  local = warp_sum(local);
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt, local);
  __syncthreads();
  const int listed = s_cnt;
  const int m = mode_only_listed ? listed : num_cards - listed;
  const int n_eff = min(n, m);
  __syncthreads();
  auto is_cand = [&](int e) -> bool {
    const bool in = (mask[e >> 5] >> (e & 31)) & 1u;
    return mode_only_listed ? in : !in;
  };

  K prefix = 0;
  bool exact_bucket = false;
  if (n_eff > 0) {
    if (threadIdx.x == 0) s_need = n_eff;
    for (int pass = 0; pass < KO::BITS / 8; ++pass) {
      const int shift = KO::BITS - 8 * (pass + 1);
      for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
      __syncthreads();
      for (int e = threadIdx.x; e < num_cards; e += blockDim.x) {
        if (!is_cand(e)) continue;
        const K key = make_key<T>(sc[e], (uint32_t)e, descending);
        if (pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8)))
          atomicAdd(&hist[int((key >> shift) & 0xff)], 1);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        int need = s_need, cum = 0, b = 255;
        for (; b > 0; --b) {
          if (cum + hist[b] >= need) break;
          cum += hist[b];
        }
        s_need = need - cum; s_digit = b; s_bucket = hist[b];
      }
      __syncthreads();
      prefix |= K((unsigned)s_digit) << shift;
      if (s_bucket == s_need) { exact_bucket = true; break; }   // whole bucket is taken
    }
  }
  (void)exact_bucket;
  // collect {key >= prefix}: exactly n_eff keys
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  if (n_eff > 0) {
    for (int e = threadIdx.x; e < num_cards; e += blockDim.x) {
      if (!is_cand(e)) continue;
      const K key = make_key<T>(sc[e], (uint32_t)e, descending);
      if (key >= prefix) {
        const int slot = atomicAdd(&s_cnt, 1);
        if (slot < n_pad) cand[slot] = key;
      }
    }
  }
  __syncthreads();
  const int got = min(s_cnt, n_pad);
  for (int i = got + threadIdx.x; i < n_pad; i += blockDim.x) cand[i] = 0;
  __syncthreads();
  // bitonic sort, descending
  for (int k = 2; k <= n_pad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const K a = cand[i], b = cand[ixj];
          const bool up = (i & k) == 0;      // "up" blocks hold larger keys first
          if (up ? (a < b) : (a > b)) { cand[i] = b; cand[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int32_t id = -1; T v = T(0);
    if (i < n_eff) {
      uint32_t t = (uint32_t)(cand[i] & 0xffffffffu);
      if (!descending) t = ~t;
      id = (int32_t)t; v = sc[id];
    }
    out_ids[int64_t(cube) * n + i] = id;
    if (out_vals) out_vals[int64_t(cube) * n + i] = v;
  }
  if (threadIdx.x == 0 && out_count) out_count[cube] = n_eff;
}

// Full ranking (n > TOPN_MAX_SMEM_N): one CTA per cube bitonic-sorts every composite key
// in a global (L2-resident) workspace of next_pow2(C) keys.
template <typename T>
__global__ void __launch_bounds__(1024)
rank_all_kernel(const T* __restrict__ scores, int64_t ld, int32_t num_cards,
                const int64_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_idx,
                int mode_only_listed, int descending, int32_t n, int32_t p2,
                typename KeyOf<T>::K* __restrict__ work, int32_t* __restrict__ out_ids, T* __restrict__ out_vals,
                int32_t* __restrict__ out_count) {
  using K = typename KeyOf<T>::K;
  extern __shared__ uint32_t mask[];
  __shared__ int s_cnt;
  const int cube = blockIdx.x;
  const T* sc = scores + int64_t(cube) * ld;
  K* keys = work + int64_t(cube) * p2;
  const int words = (num_cards + 31) >> 5;
  for (int w = threadIdx.x; w < words; w += blockDim.x) mask[w] = 0;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  for (int64_t p = mask_ptr[cube] + threadIdx.x; p < mask_ptr[cube + 1]; p += blockDim.x) {
    const int32_t c = mask_idx[p];
    if (c >= 0 && c < num_cards) atomicOr(&mask[c >> 5], 1u << (c & 31));
  }
  __syncthreads();
  int local = 0;
  for (int e = threadIdx.x; e < p2; e += blockDim.x) {
    K key = 0;
    if (e < num_cards) {
      const bool in = (mask[e >> 5] >> (e & 31)) & 1u;
      if (mode_only_listed ? in : !in) { key = make_key<T>(sc[e], (uint32_t)e, descending); ++local; }
    }
    keys[e] = key;
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt, local);
  __syncthreads();
  const int n_eff = min(n, s_cnt);
  for (int k = 2; k <= p2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < p2; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const K a = keys[i], b = keys[ixj];
          const bool up = (i & k) == 0;
          if (up ? (a < b) : (a > b)) { keys[i] = b; keys[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int32_t id = -1; T v = T(0);
    if (i < n_eff) {
      uint32_t t = (uint32_t)(keys[i] & 0xffffffffu);
      if (!descending) t = ~t;
      id = (int32_t)t; v = sc[id];
    }
    out_ids[int64_t(cube) * n + i] = id;
    if (out_vals) out_vals[int64_t(cube) * n + i] = v;
  }
  if (threadIdx.x == 0 && out_count) out_count[cube] = n_eff;
}

// ------------------------------------------------------------- warp-per-cube streaming select (float32, n <= 128)
// One pass over the scores: a warp keeps the best keys seen so far in a 256-slot shared buffer and a running
// threshold (the n-th best key); a score only enters the buffer when its composite key beats the threshold,
// and the buffer is sorted and cut back to n whenever it fills.  After the first few hundred elements almost
// nothing passes (expected insertions ~ n ln(C/n)), so the kernel is one coalesced read of the row plus a
// handful of 256-key bitonic sorts -- against up to eight passes with shared-memory histogram atomics in the
// radix-select kernel above.  Same total order (score, then index) => identical ids.
constexpr int WS_WARPS = 8;
constexpr int WS_CAP = 256;
constexpr int WS_MAX_N = 128;

__device__ __forceinline__ void warp_bitonic_desc(unsigned long long* buf, int lane) {
  for (int k = 2; k <= WS_CAP; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int t = 0; t < WS_CAP / 64; ++t) {
        const int p = lane + 32 * t;                              // compare-exchange pair index
        const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));      // element with bit j clear
        const int x = i | j;
        const unsigned long long a = buf[i], b = buf[x];
        const bool up = (i & k) == 0;                             // "up" blocks hold larger keys first
        if (up ? (a < b) : (a > b)) { buf[i] = b; buf[x] = a; }
      }
      __syncwarp();
    }
  }
}

template <bool SIGMOID>
__global__ void __launch_bounds__(WS_WARPS * 32)
topn_warpselect_kernel(const float* __restrict__ scores, int64_t ld, int32_t num_cards, int32_t batch,
                       const int64_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_idx,
                       int mode_only_listed, int descending, int32_t n, int32_t* __restrict__ out_ids,
                       float* __restrict__ out_vals, int32_t* __restrict__ out_count) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int words = (num_cards + 31) >> 5;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(smem_raw) + warp * WS_CAP;
  uint32_t* mask = reinterpret_cast<uint32_t*>(smem_raw + size_t(WS_WARPS) * WS_CAP * 8) + size_t(warp) * words;
  const int cube = blockIdx.x * WS_WARPS + warp;
  if (cube >= batch) return;                    // warps are independent: no CTA-wide barrier below
  for (int w = lane; w < words; w += 32) mask[w] = 0;
  __syncwarp();
  const int64_t mb = mask_ptr[cube], me = mask_ptr[cube + 1];
  for (int64_t p = mb + lane; p < me; p += 32) {
    const int32_t c = mask_idx[p];
    if (c >= 0 && c < num_cards) atomicOr(&mask[c >> 5], 1u << (c & 31));
  }
  __syncwarp();
  int listed = 0;
  for (int w = lane; w < words; w += 32) listed += __popc(mask[w]);
  listed = warp_sum(listed);
  const int m = mode_only_listed ? listed : num_cards - listed;
  const int n_eff = min(n, m);
  const float* sc = scores + int64_t(cube) * ld;
  unsigned long long thr = 0;                   // keys must beat this to enter the buffer
  int cnt = 0;                                  // live keys in buf (warp-uniform)
  // zbound: a bound on the RAW value that lets almost every element skip the key (and, fused, the sigmoid: expf +
  // division) altogether.  Plain scores: the threshold's own score (ties still go through the exact key compare).
  // SIGMOID: keys are
  // built from float32 sigmoid(z) so that saturated scores tie exactly as in the reference; sigmoid is monotone, so
  // an element can only beat the threshold score p_thr if z lies on the right side of logit(p_thr).  The bound is
  // taken 1e-6 relative (~16 float32 ulps) on the safe side of p_thr, which covers the few-ulp error of sigmoid_f32:
  // no element whose key would enter the buffer is ever rejected.  (NaN logits fail the test and are skipped.)
  float zbound = descending ? -INFINITY : INFINITY;

  auto prune = [&]() {
    __syncwarp();
    for (int i = cnt + lane; i < WS_CAP; i += 32) buf[i] = 0;
    __syncwarp();
    warp_bitonic_desc(buf, lane);
    if (cnt >= n_eff && n_eff > 0) {
      thr = buf[n_eff - 1]; cnt = n_eff;
      uint32_t u = (uint32_t)(thr >> 32);
      if (!descending) u = ~u;
      const float pthr = __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);   // the threshold's score
      if (!SIGMOID) {
        zbound = pthr;        // a raw score can only enter if it is >= (descending) / <= (ascending) the threshold score
      } else {
        const double p = double(pthr);
        if (descending) {
          const double pm = p * (1.0 - 1e-6) - 1e-40;
          zbound = pm <= 0.0 ? -INFINITY : float(log(pm / (1.0 - pm))) - 1e-3f;
        } else {
          const double pp = p * (1.0 + 1e-6) + 1e-40;
          zbound = pp >= 1.0 ? INFINITY : float(log(pp / (1.0 - pp))) + 1e-3f;
        }
      }
    }
  };

  // `zbound` pre-filter: the cheap test every element takes; only survivors build a key (and, fused, a sigmoid)
  auto maybe = [&](float x) -> bool { return descending ? x >= zbound : x <= zbound; };
  auto offer = [&](bool c, float x, int e) {           // warp-collective: insert the lanes' surviving candidates
    unsigned long long key = 0;
    if (c) key = make_key<float>(SIGMOID ? sigmoid_f32(x) : x, (uint32_t)e, descending);
    const bool pass = key > thr;
    const unsigned bal = __ballot_sync(0xffffffffu, pass);
    if (bal) {
      if (pass) buf[cnt + __popc(bal & ((1u << lane) - 1u))] = key;
      cnt += __popc(bal);
      if (cnt > WS_CAP - 32) prune();
    }
  };
  const bool vec = (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(scores) & 15) == 0;
  if (n_eff > 0 && vec) {
    // 16-byte loads: a lane takes 4 consecutive scores (and the 4 matching mask bits), two loads in flight; when none
    // of the warp's 256 elements survives the pre-filter -- the steady state after the first few hundred elements --
    // the iteration is two loads, eight compares and one vote
    for (int base = 0; base < num_cards; base += 256) {
      float4 q[2];
      uint32_t mb[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int e0 = base + 128 * u + 4 * lane;
        uint32_t bits = 0u;
        if (e0 < num_cards) {
          bits = (mask[e0 >> 5] >> (e0 & 31)) & 0xfu;
          if (!mode_only_listed) bits ^= 0xfu;
          if (e0 + 3 >= num_cards) bits &= (1u << (num_cards - e0)) - 1u;      // ragged end of the row
        }
        mb[u] = bits;
        q[u] = bits ? ld_nc_f4(sc + e0) : make_float4(0.f, 0.f, 0.f, 0.f);      // e0 + 3 < ld (ld % 4 == 0)
      }
      bool c[2][4];
      bool any = false;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float x[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { c[u][j] = ((mb[u] >> j) & 1u) && maybe(x[j]); any |= c[u][j]; }
      }
      if (!__any_sync(0xffffffffu, any)) continue;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float x[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // re-test against the bound: it may have tightened since the flags were computed (a prune in between);
          // usually one lane of one (u, j) slot survives, the other seven slots cost a single vote
          const bool cc = c[u][j] && maybe(x[j]);
          if (!__any_sync(0xffffffffu, cc)) continue;
          offer(cc, x[j], base + 128 * u + 4 * lane + j);
        }
      }
    }
    prune();
  } else if (n_eff > 0) {
    for (int base = 0; base < num_cards; base += 128) {
      float v[4];
      bool cand[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {               // four independent 128-byte row segments in flight
        const int e = base + 32 * u + lane;
        const int wi = (base >> 5) + u;
        const uint32_t mw = wi < words ? mask[wi] : 0u;
        cand[u] = e < num_cards && ((((mw >> lane) & 1u) != 0) == (mode_only_listed != 0));
        v[u] = cand[u] ? sc[e] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) offer(cand[u] && maybe(v[u]), v[u], base + 32 * u + lane);
    }
    prune();
  }
  __syncwarp();
  for (int i = lane; i < n; i += 32) {
    int32_t id = -1; float val = 0.f;
    if (i < n_eff) {
      const unsigned long long key = buf[i];
      uint32_t t = (uint32_t)(key & 0xffffffffu), u = (uint32_t)(key >> 32);
      if (!descending) { t = ~t; u = ~u; }
      id = (int32_t)t;
      val = __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);      // inverse of KeyOf<float>::ord
    }
    out_ids[int64_t(cube) * n + i] = id;
    if (out_vals) out_vals[int64_t(cube) * n + i] = val;
  }
  if (lane == 0 && out_count) out_count[cube] = n_eff;
}

template <bool SIGMOID>
static int warpselect_launch(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                             const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n,
                             int32_t* out_ids, float* out_vals, int32_t* out_count, cudaStream_t st) {
  const size_t smem = size_t(WS_WARPS) * (WS_CAP * 8 + size_t((num_cards + 31) / 32) * 4);
  CC_REQUIRE(smem <= 200 * 1024, "cc_topn_masked: C=%d needs %zu bytes of shared memory", num_cards, smem);
  if (smem > 48 * 1024)
    CC_CHECK_CUDA(cudaFuncSetAttribute(topn_warpselect_kernel<SIGMOID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  topn_warpselect_kernel<SIGMOID><<<ceil_div(batch, WS_WARPS), WS_WARPS * 32, smem, st>>>(
      scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, descending, n, out_ids, out_vals, out_count);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// ------------------------------------------------------------- CTA-per-cube row select (float32, n <= 128)
// The HBM-bound form of the select.  Persistent CTAs walk the cubes; each cube's score row (4C bytes, 83.5 KB at
// C = 20 884) is pulled into shared memory by bulk asynchronous copies (cp.async.bulk, completion on an mbarrier), so
// no thread ever waits on a global load of scores and the next row streams in from HBM while this one is ranked (two
// CTAs per SM with one row buffer each, or one CTA with two buffers).  Ranking a resident row takes two sweeps of it:
//   sweep 1  every thread keeps the extreme of its float4 stride (one compare per four elements); four neighbouring
//            threads merge to one of 128 leaders; the leaders are ranked by counting on 32-bit stand-ins and the n-th
//            largest, low bits cleared, becomes the threshold T.  T is a lower bound of the key of a real element with
//            at least n elements at or above it, so the answer's last key is >= T; with the row spread over 128 leader
//            strides only ~1.3 n elements lie above it (n = 50: ~63).
//   sweep 2  the elements that pass the raw-value bound of T (one float compare per group of four) are appended raw
//            to a small buffer, keyed one survivor per thread, ranked against each other by counting, and written at
//            their rank.
// Masked cards are overwritten with a NaN sentinel in the shared copy of the row (every compare with it is false), so
// the sweeps carry no mask test.  If an adversarial row leaves more than RS_CAP survivors, T is raised to the n-th
// largest of the first RS_CAP of them (again a valid bound, strictly tighter) and sweep 2 is repeated with the exact key
// test.  Same total order on (score, index) as the two kernels above => identical ids.  NaN scores are never selected.
// The selection logic is restated on the host in tests/rowselect_model.py (DESIGN.md 4a).
constexpr int RS_THREADS = 512;
constexpr int RS_CAP = 1024;
constexpr int RS_LEADERS = 128;
constexpr uint32_t RS_SENTINEL = 0x7fc0babeu;      // quiet NaN with a payload no arithmetic produces
constexpr uint32_t RS_COPY_BYTES = 16384;          // one bulk copy; a row is a handful of them on one barrier
static_assert(RS_THREADS == 4 * RS_LEADERS, "rs_rank_partial splits the compare range into RS_THREADS / RS_LEADERS = 4 parts");

__device__ __forceinline__ uint32_t rs_smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void rs_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rs_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void rs_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(rs_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rs_mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = rs_smem_u32(bar);
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    if (done) break;
    if (++spins > (1u << 26)) __trap();            // watchdog: a protocol bug must not hang the GPU
  }
}
__device__ __forceinline__ void rs_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(rs_smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(rs_smem_u32(bar)) : "memory");
}

// rk[i] += #{ j in this thread's quarter of [0, m) : keys[j] > keys[i] }.  The caller zeroes rk[0, m) and
// synchronises before, and synchronises after; then rk[i] is the rank of keys[i] (0 = largest).  The inner loop reads
// one key per iteration for the whole warp (a broadcast), so it is conflict-free.
__device__ __forceinline__ void rs_rank_partial(const unsigned long long* keys, int m, int* rk, int tid) {
  const int g = tid & (RS_LEADERS - 1), q = tid / RS_LEADERS;
  const int chunk = (m + 3) >> 2;
  const int j0 = q * chunk, j1 = min(m, j0 + chunk);
  for (int i = g; i < m; i += RS_LEADERS) {
    const unsigned long long mine = keys[i];
    int c = 0;
    for (int j = j0; j < j1; ++j) c += (keys[j] > mine) ? 1 : 0;
    if (c) atomicAdd(&rk[i], c);
  }
}

// The 128 merged leaders are ranked on 32-bit stand-ins: the score word of the key with its 7 low bits replaced by the
// leader's number (unique, so ranks are a permutation; one compare is a single integer test).  The stand-in order can
// differ from the key order only between leaders whose score words agree in all but the 7 low bits, so the threshold
// is taken with those bits cleared: every leader that ranks at or above the chosen one still has key >= T.
__device__ __forceinline__ void rs_rank32_partial(const uint32_t* a, int* rk, int tid) {
  const int g = tid & (RS_LEADERS - 1), q = tid / RS_LEADERS;
  const uint32_t mine = a[g];
  const uint4* a4 = reinterpret_cast<const uint4*>(a) + q * (RS_LEADERS / 16);
  int c = 0;
#pragma unroll
  for (int j = 0; j < RS_LEADERS / 16; ++j) {
    const uint4 w = a4[j];
    c += (w.x > mine) + (w.y > mine) + (w.z > mine) + (w.w > mine);
  }
  if (c) atomicAdd(&rk[g], c);
}

// PROF: thread 0 accumulates clock64() deltas per phase and writes them to prof[blockIdx.x][RS_PROF_SLOTS] (diagnostic
// instantiation behind cc_topn_rowselect_profile; the product instantiations compile the stamps out)
//
// REGS (cc_topn_set_algo(4); for rows that fit RS_GROUPS float4 per thread): the ncu source view of the kernel without
// it (profiles/r02/topn_rowselect_stalls.txt) shows where a cube's ~14 000 cycles go -- 3% waiting for the row (HBM), 32%
// in sweep 2 (branch-resolve and shared-memory-atomic stalls of the diverged push path, entered anew for every float4
// group that holds a survivor), 25% at barriers behind the slowest warp of a sweep.  REGS keeps the per-group extremes
// of sweep 1 in registers (11 floats), so sweep 2 re-reads NOTHING from shared memory: it is 11 predicated register
// compares per thread that leave a bit mask of the groups to look at again.  The ~70 threads of 512 whose mask is not
// empty then enter ONE diverged block per warp (fetch the group, append each survivor already keyed -- sigmoid
// included -- with one shared-memory atomic), instead of one excursion per group.  Both counting ranks (the 128 leaders,
// the ~70 survivors) are summed over four NEIGHBOURING lanes with shuffles: no rank array, no atomics, and the thread
// that holds a rank acts on it directly -- four barriers per cube instead of nine.  The survivor counter alternates
// between two words so that its reset needs no barrier of its own.  More than RS_CAP survivors (adversarial rows) and
// the only-listed mode take the path of the kernel without REGS, which keeps its own overflow handling.
constexpr int RS_PROF_SLOTS = 10;
constexpr int RS_GROUPS = 11;                      // float4 groups per thread held in registers: C <= 4 * 11 * 512 = 22 528
template <bool SIGMOID, bool DESC, bool PROF = false, bool REGS = false>
__global__ void __launch_bounds__(RS_THREADS, 2)
topn_rowselect_kernel(const float* __restrict__ scores, int64_t ld, int32_t num_cards, int32_t batch,
                      const int64_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_idx,
                      int mode_only_listed, int32_t n, int nbuf, int32_t* __restrict__ out_ids,
                      float* __restrict__ out_vals, int32_t* __restrict__ out_count, long long* __restrict__ prof = nullptr) {
  long long acc[RS_PROF_SLOTS] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  long long tprev = 0;
  auto stamp = [&](int slot) {
    if constexpr (PROF) {
      if (threadIdx.x == 0) { const long long t = clock64(); acc[slot] += t - tprev; tprev = t; }
    }
  };
  if constexpr (PROF) tprev = clock64();
  // (nvcc warns that the other kernels of this file declare the array with 16-byte alignment: harmless, and left alone
  // because the build that was verified on the GPU has it)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar[2];
  __shared__ unsigned long long s_T;
  __shared__ float s_zb;
  __shared__ int s_cnt;
  __shared__ int s_cnt2[2];                                 // REGS: the survivor counter of even / odd cubes
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int cr = (num_cards + 3) & ~3;                      // row length in shared memory (<= ld: ld % 4 == 0)
  const int cr4 = cr >> 2;
  const uint32_t row_bytes = uint32_t(cr) * 4u;
  const int words = (num_cards + 31) >> 5;
  float* const row_base = reinterpret_cast<float*>(smem_raw);                                              // nbuf rows of cr floats
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw + size_t(nbuf) * row_bytes);   // RS_CAP
  uint32_t* lead32 = reinterpret_cast<uint32_t*>(keys);            // the leaders' stand-ins live here before sweep 2
  int* rk = reinterpret_cast<int*>(keys + RS_CAP);                                                        // RS_CAP, zero between uses
  uint32_t* bm = reinterpret_cast<uint32_t*>(rk + RS_CAP);                                                // words
  constexpr float WORST = DESC ? -INFINITY : INFINITY;

  auto issue = [&](int cube, int b) {                       // one thread: the whole row on barrier b
    const char* src = reinterpret_cast<const char*>(scores + int64_t(cube) * ld);
    char* dst = reinterpret_cast<char*>(row_base + size_t(b) * cr);
    rs_mbar_expect_tx(&bar[b], row_bytes);
    for (uint32_t off = 0; off < row_bytes; off += RS_COPY_BYTES)
      rs_bulk_g2s(dst + off, src + off, min(RS_COPY_BYTES, row_bytes - off), &bar[b]);
  };

  const int stride = gridDim.x;
  const int cube0 = blockIdx.x;
  if (tid == 0) {
    rs_mbar_init(&bar[0], 1);
    rs_mbar_init(&bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    s_cnt = 0; s_T = 0ull; s_zb = WORST; s_cnt2[0] = 0; s_cnt2[1] = 0;
  }
  for (int i = tid; i < RS_CAP; i += RS_THREADS) rk[i] = 0;
  __syncthreads();
  if (tid == 0) {
    for (int b = 0; b < nbuf; ++b)
      if (cube0 + b * stride < batch) issue(cube0 + b * stride, b);
  }
  // The mask list of a cube is read through registers: its first two entries per thread are loaded one cube ahead and
  // its (begin, end) pair two cubes ahead, so their global-memory latency hides behind the previous cube's sweeps.
  int64_t mb = 0, me = 0, mb1 = 0, me1 = 0;
  int32_t c0 = -1, c1 = -1;
  if (cube0 < batch) {
    mb = mask_ptr[cube0]; me = mask_ptr[cube0 + 1];
    if (mb + tid < me) c0 = mask_idx[mb + tid];
    if (mb + tid + RS_THREADS < me) c1 = mask_idx[mb + tid + RS_THREADS];
  }
  if (cube0 + stride < batch) { mb1 = mask_ptr[cube0 + stride]; me1 = mask_ptr[cube0 + stride + 1]; }

  auto pass = [&](float x, float zb) -> bool { return DESC ? x >= zb : x <= zb; };
  // survivors are stored raw (score bits, index); their keys are made afterwards, one survivor per thread, instead of
  // one sigmoid at a time in a diverged warp.  exact = 0 keeps every element that passes the raw-value bound (a superset
  // of {key >= T}: the final ranking is exact anyway); exact = 1 (after an overflow) tests the key itself.
  auto push = [&](float x, int e, unsigned long long T, bool exact) {
    if (exact && make_key<float>(SIGMOID ? sigmoid_f32(x) : x, (uint32_t)e, DESC) < T) return;
    const unsigned long long raw = ((unsigned long long)__float_as_uint(x) << 32) | (unsigned long long)(uint32_t)e;
    const int slot = atomicAdd(&s_cnt, 1);
    if (slot < RS_CAP) keys[slot] = raw;
  };
  auto raw_to_key = [&](unsigned long long raw) {
    const float x = __uint_as_float((uint32_t)(raw >> 32));
    return make_key<float>(SIGMOID ? sigmoid_f32(x) : x, (uint32_t)(raw & 0xffffffffu), DESC);
  };
  const uint32_t lt_mask = (1u << lane) - 1u;

  int it = 0;
  for (int cube = cube0; cube < batch; cube += stride, ++it) {
    const int b = nbuf == 2 ? (it & 1) : 0;
    const uint32_t parity = uint32_t(nbuf == 2 ? (it >> 1) : it) & 1u;
    float* row = row_base + size_t(b) * cr;
    const float4* row4 = reinterpret_cast<const float4*>(row);
    int32_t nc0 = -1, nc1 = -1;
    int64_t mb2 = 0, me2 = 0;
    if (cube + stride < batch) {
      if (mb1 + tid < me1) nc0 = mask_idx[mb1 + tid];
      if (mb1 + tid + RS_THREADS < me1) nc1 = mask_idx[mb1 + tid + RS_THREADS];
    }
    if (cube + 2 * stride < batch) { mb2 = mask_ptr[cube + 2 * stride]; me2 = mask_ptr[cube + 2 * stride + 1]; }
    stamp(0);
    auto for_each_listed = [&](auto&& f) {
      f(c0); f(c1);
      for (int64_t p = mb + 2 * RS_THREADS + tid; p < me; p += RS_THREADS) f(mask_idx[p]);
    };
    rs_mbar_wait(&bar[b], parity);
    stamp(1);                                               // 0: loop top + prefetch (stamped below), 1: wait for the row

    float gmax[RS_GROUPS];                                  // REGS: extreme of each of this thread's float4 groups
    if (!mode_only_listed) {
      // masked cards (and the up to three floats of row padding) -> sentinel
      for_each_listed([&](int32_t c) { if (c >= 0 && c < num_cards) reinterpret_cast<uint32_t*>(row)[c] = RS_SENTINEL; });
      if (tid < cr - num_cards) reinterpret_cast<uint32_t*>(row)[num_cards + tid] = RS_SENTINEL;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // before the next bulk copy overwrites them
      __syncthreads();
      stamp(2);                                             // 2: sentinels + fence + barrier
      // sweep 1: the best element of this thread's float4 stride.  Per group of four only its extreme is compared
      // (NaN sentinels drop out of fmaxf / fminf); the winner's position inside its group is resolved afterwards, to
      // the index the total order prefers among equal scores (descending: the largest, ascending: the smallest).
      float best = WORST;
      int bv = -1;
      if constexpr (REGS) {
#pragma unroll
        for (int j = 0; j < RS_GROUPS; ++j) {
          const int v = tid + j * RS_THREADS;
          float g = DESC ? -INFINITY : INFINITY;
          if (v < cr4) {
            const float4 q = row4[v];
            g = DESC ? fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)) : fminf(fminf(q.x, q.y), fminf(q.z, q.w));
            if (DESC ? g >= best : g < best) { best = g; bv = v; }
          }
          gmax[j] = g;
        }
      } else {
        for (int v = tid; v < cr4; v += RS_THREADS) {
          const float4 q = row4[v];
          if (DESC) { const float g = fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)); if (g >= best) { best = g; bv = v; } }
          else      { const float g = fminf(fminf(q.x, q.y), fminf(q.z, q.w)); if (g < best) { best = g; bv = v; } }
        }
      }
      stamp(3);                                             // 3: sweep 1
      unsigned long long k = 0ull;
      if (bv >= 0) {
        const float4 q = row4[bv];
        const int j = DESC ? (q.w == best ? 3 : q.z == best ? 2 : q.y == best ? 1 : 0)
                           : (q.x == best ? 0 : q.y == best ? 1 : q.z == best ? 2 : 3);
        k = make_key<float>(SIGMOID ? sigmoid_f32(best) : best, (uint32_t)(4 * bv + j), DESC);
      }
      {                                                     // four neighbouring threads -> one leader
        unsigned long long o = __shfl_xor_sync(0xffffffffu, k, 1); k = o > k ? o : k;
        o = __shfl_xor_sync(0xffffffffu, k, 2); k = o > k ? o : k;
      }
      if ((lane & 3) == 0) lead32[tid >> 2] = ((uint32_t)(k >> 32) & ~0x7fu) | (uint32_t)(tid >> 2);
      __syncthreads();
      // score words at or below the code of the worst infinity (its low bits cleared would decode to a NaN): no bound
      auto publish = [&](uint32_t stand_in) {
        const uint32_t uw = stand_in & ~0x7fu;
        const unsigned long long t = uw > 0x007fffffu ? (unsigned long long)uw << 32 : 0ull;
        s_T = t; s_zb = rs_raw_bound<SIGMOID>(t, DESC);
      };
      if constexpr (REGS) {
        // leader tid / 4 against quarter tid % 4 of the stand-ins; the four partial counts meet by shuffles
        // (the quarters are 128 bytes apart, i.e. in the same banks: each starts two 16-byte words further into its
        // quarter, so the four addresses of an 8-lane load phase fall into different bank groups)
        const uint32_t mine = lead32[tid >> 2];
        const int q = tid & 3;
        const uint4* a4 = reinterpret_cast<const uint4*>(lead32) + q * (RS_LEADERS / 16);
        int c = 0;
#pragma unroll
        for (int j = 0; j < RS_LEADERS / 16; ++j) {
          const uint4 w = a4[(j + 2 * q) & (RS_LEADERS / 16 - 1)];
          c += (w.x > mine) + (w.y > mine) + (w.z > mine) + (w.w > mine);
        }
        c += __shfl_xor_sync(0xffffffffu, c, 1);
        c += __shfl_xor_sync(0xffffffffu, c, 2);
        if ((tid & 3) == 0 && c == n - 1) publish(mine);
        if (tid == 0) s_cnt2[(it + 1) & 1] = 0;             // the next cube's counter (last read behind the previous cube's barriers)
      } else {
        rs_rank32_partial(lead32, rk, tid);
        __syncthreads();
        if (tid < RS_LEADERS) {
          if (rk[tid] == n - 1) publish(lead32[tid]);
          rk[tid] = 0;
        }
      }
      __syncthreads();
      stamp(4);                                             // 4: leaders: keys, merge, ranking, threshold
    }

    int m = 0;
    if constexpr (REGS) {
      if (!mode_only_listed) {
        // sweep 2 over registers: which of this thread's groups hold an element at or above the bound
        const float zb = s_zb;
        int* const cnt = &s_cnt2[it & 1];
        uint32_t hits = 0u;
#pragma unroll
        for (int j = 0; j < RS_GROUPS; ++j) hits |= pass(gmax[j], zb) ? (1u << j) : 0u;
        while (hits) {                                      // ~1 thread in 7 enters, nearly always for one group
          const int j = __ffs(hits) - 1;
          hits &= hits - 1u;
          const int v = tid + j * RS_THREADS;
          if (v < cr4) {                                    // (a bound of -inf / +inf also passes the groups beyond the row)
            const float4 q = row4[v];
            uint32_t em = (pass(q.x, zb) ? 1u : 0u) | (pass(q.y, zb) ? 2u : 0u) | (pass(q.z, zb) ? 4u : 0u) | (pass(q.w, zb) ? 8u : 0u);
            while (em) {                                    // one instance of the push code, nearly always run once
              const int e = __ffs(em) - 1;
              em &= em - 1u;
              const float x = e == 0 ? q.x : e == 1 ? q.y : e == 2 ? q.z : q.w;
              const int slot = atomicAdd(cnt, 1);
              if (slot < RS_CAP) keys[slot] = ((unsigned long long)__float_as_uint(x) << 32) | (unsigned long long)(uint32_t)(4 * v + e);
            }
          }
        }
        __syncthreads();
        m = *cnt;
        stamp(5);                                           // 5: sweep 2, raw survivors appended (+ barrier)
        // raw survivors -> composite keys, one per thread (a sigmoid each: three warps' worth instead of a few lanes of all 16)
        if (tid < min(m, RS_CAP)) keys[tid] = raw_to_key(keys[tid]);
        if (tid + RS_THREADS < min(m, RS_CAP)) keys[tid + RS_THREADS] = raw_to_key(keys[tid + RS_THREADS]);
        // the final ranking reads four equal, even-sized quarters of the keys: zero keys (nothing ranks below them) fill
        // the up to seven slots behind the last one (past RS_CAP they land on the zeroed rank array: harmless)
        const int chunk = (((min(m, RS_CAP) + 3) >> 2) + 1) & ~1;
        if (tid >= RS_THREADS - 8 && m <= RS_CAP && m + (tid - (RS_THREADS - 8)) < 4 * chunk) keys[m + (tid - (RS_THREADS - 8))] = 0ull;
        __syncthreads();
        stamp(6);                                           // 6: survivors -> keys (+ barrier)
        if (m <= RS_CAP) {
          // the row is not needed any more; the last warp has no ranking work unless m > 120
          if (tid == RS_THREADS - 32 && cube + nbuf * stride < batch) issue(cube + nbuf * stride, b);
          // survivor base + tid / 4 against quarter tid % 4 of the keys; the thread that holds the rank writes the result
          // (every quarter holds `chunk` keys, read two at a time: the same trip count for every thread)
          const ulonglong2* k2 = reinterpret_cast<const ulonglong2*>(keys) + (tid & 3) * (chunk >> 1);
          for (int base = 0; base < m; base += RS_LEADERS) {
            const int i = base + (tid >> 2);
            const unsigned long long mine = i < m ? keys[i] : ~0ull;
            int c = 0;
#pragma unroll 4
            for (int j = 0; j < (chunk >> 1); ++j) {
              const ulonglong2 w = k2[j];
              c += ((w.x > mine) ? 1 : 0) + ((w.y > mine) ? 1 : 0);
            }
            c += __shfl_xor_sync(0xffffffffu, c, 1);
            c += __shfl_xor_sync(0xffffffffu, c, 2);
            if (i < m && (tid & 3) == 0 && c < n) {
              uint32_t t = (uint32_t)(mine & 0xffffffffu), u = (uint32_t)(mine >> 32);
              if (!DESC) { t = ~t; u = ~u; }
              out_ids[int64_t(cube) * n + c] = (int32_t)t;
              if (out_vals) out_vals[int64_t(cube) * n + c] = __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
            }
          }
          stamp(7);                                         // 7: issue of the next row + final ranking + write-out
          for (int i = m + tid; i < n; i += RS_THREADS) {
            out_ids[int64_t(cube) * n + i] = -1;
            if (out_vals) out_vals[int64_t(cube) * n + i] = 0.f;
          }
          if (tid == 0 && out_count) out_count[cube] = min(n, m);
          mb = mb1; me = me1; c0 = nc0; c1 = nc1; mb1 = mb2; me1 = me2;
          stamp(8);
          continue;
        }
      }
    }
    // sweep 2 over the shared row (the kernel without REGS; with REGS: only-listed mode and cubes whose survivors
    // number more than RS_CAP), repeated with a raised threshold if more than RS_CAP elements survive
    for (int round = 0;; ++round) {
      if (mode_only_listed) {
        for (int w = tid; w < words; w += RS_THREADS) bm[w] = 0u;
        __syncthreads();
      }
      const unsigned long long T = s_T;                     // (read behind this cube's first barrier)
      const float zb = s_zb;
      const bool exact = round > 0;
      if (mode_only_listed) {
        for_each_listed([&](int32_t c) {
          if (c < 0 || c >= num_cards) return;
          const uint32_t bit = 1u << (c & 31);
          if (atomicOr(&bm[c >> 5], bit) & bit) return;             // duplicate entry of the list
          const float x = row[c];
          if (pass(x, zb)) push(x, c, T, exact);
        });
      } else {
        for (int v = tid; v < cr4; v += RS_THREADS) {
          const float4 q = row4[v];
          const float g = DESC ? fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)) : fminf(fminf(q.x, q.y), fminf(q.z, q.w));
          if (pass(g, zb)) {
            if (pass(q.x, zb)) push(q.x, 4 * v, T, exact);
            if (pass(q.y, zb)) push(q.y, 4 * v + 1, T, exact);
            if (pass(q.z, zb)) push(q.z, 4 * v + 2, T, exact);
            if (pass(q.w, zb)) push(q.w, 4 * v + 3, T, exact);
          }
        }
      }
      __syncthreads();
      m = s_cnt;
      stamp(5);                                             // 5: sweep 2 (+ barrier)
      // raw survivors -> composite keys (each thread its own slots)
      for (int i = tid; i < min(m, RS_CAP); i += RS_THREADS) keys[i] = raw_to_key(keys[i]);
      __syncthreads();
      stamp(6);                                             // 6: survivors -> keys (+ barrier)
      if (m <= RS_CAP) break;
      // overflow: T <- n-th largest of the RS_CAP survivors kept (n <= 128 < RS_CAP), then sweep again, exactly
      rs_rank_partial(keys, RS_CAP, rk, tid);
      __syncthreads();
      if (tid == 0) s_cnt = 0;
      for (int i = tid; i < RS_CAP; i += RS_THREADS) {
        if (rk[i] == n - 1) { const unsigned long long t = keys[i]; s_T = t; s_zb = rs_raw_bound<SIGMOID>(t, DESC); }
        rk[i] = 0;
      }
      __syncthreads();
    }
    // the row is not needed any more: its buffer takes the row of the cube nbuf turns ahead while this one is ranked
    if (tid == 0 && cube + nbuf * stride < batch) issue(cube + nbuf * stride, b);

    // rank the m survivors among themselves and write the first n at their rank
    auto write_ranked = [&](unsigned long long key, int r) {
      uint32_t t = (uint32_t)(key & 0xffffffffu), u = (uint32_t)(key >> 32);
      if (!DESC) { t = ~t; u = ~u; }
      out_ids[int64_t(cube) * n + r] = (int32_t)t;
      if (out_vals) out_vals[int64_t(cube) * n + r] = __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
    };
    rs_rank_partial(keys, m, rk, tid);
    __syncthreads();
    stamp(7);                                               // 7: issue of the next row + final ranking (+ barrier)
    // every thread has read s_cnt, s_T and s_zb by now; their next use lies behind the next cube's barriers
    if (tid == 0) { s_cnt = 0; s_T = 0ull; s_zb = WORST; }
    for (int i = tid; i < m; i += RS_THREADS) {
      const int r = rk[i];
      rk[i] = 0;
      if (r < n) write_ranked(keys[i], r);
    }
    for (int i = m + tid; i < n; i += RS_THREADS) {
      out_ids[int64_t(cube) * n + i] = -1;
      if (out_vals) out_vals[int64_t(cube) * n + i] = 0.f;
    }
    if (tid == 0 && out_count) out_count[cube] = min(n, m);
    mb = mb1; me = me1; c0 = nc0; c1 = nc1; mb1 = mb2; me1 = me2;
    stamp(8);                                               // 8: write-out
  }
  if constexpr (PROF) {
    if (threadIdx.x == 0 && prof) {
      acc[9] = it;                                          // cubes this CTA ranked
      for (int i = 0; i < RS_PROF_SLOTS; ++i) prof[int64_t(blockIdx.x) * RS_PROF_SLOTS + i] = acc[i];
    }
  }
}

static size_t rowselect_smem_bytes(int32_t num_cards, int nbuf) {
  const size_t cr = (size_t(num_cards) + 3) & ~size_t(3);
  return size_t(nbuf) * cr * 4 + size_t(RS_CAP) * 8 + size_t(RS_CAP) * 4 + size_t((num_cards + 31) / 32) * 4;
}

// rows must be 16-byte aligned and a whole number of 16-byte units (bulk copies), and two of them must fit in shared memory
static bool rowselect_eligible(const float* scores, int64_t ld, int32_t num_cards, int32_t n) {
  return n <= WS_MAX_N && (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(scores) & 15) == 0 &&
         rowselect_smem_bytes(num_cards, 2) + 1024 <= 227 * 1024;
}

// variant 0: one CTA per SM, two row buffers; variant 1: two CTAs per SM, one row buffer each; variant 2: the REGS form
// of the kernel (group maxima in registers, ballot-compacted survivors) in the launch shape of variant 1
template <bool SIGMOID, bool DESC>
static int rowselect_launch_t(int variant, const float* scores, int64_t ld, int32_t num_cards, int32_t batch,
                              const int64_t* mask_ptr, const int32_t* mask_idx, int mode_only_listed, int32_t n,
                              int32_t* out_ids, float* out_vals, int32_t* out_count, cudaStream_t st) {
  const int nbuf = variant == 0 ? 2 : 1, ctas = variant == 0 ? 1 : 2;
  const size_t smem = rowselect_smem_bytes(num_cards, nbuf);
  const int grid = batch < ctas * sm_count() ? batch : ctas * sm_count();
  if (variant == 2) {
    CC_CHECK_CUDA(cudaFuncSetAttribute(topn_rowselect_kernel<SIGMOID, DESC, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_rowselect_kernel<SIGMOID, DESC, false, true><<<grid, RS_THREADS, smem, st>>>(
        scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, n, nbuf, out_ids, out_vals, out_count);
  } else {
    CC_CHECK_CUDA(cudaFuncSetAttribute(topn_rowselect_kernel<SIGMOID, DESC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_rowselect_kernel<SIGMOID, DESC><<<grid, RS_THREADS, smem, st>>>(
        scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, n, nbuf, out_ids, out_vals, out_count);
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

template <bool SIGMOID>
static int rowselect_launch(int variant, const float* scores, int64_t ld, int32_t num_cards, int32_t batch,
                            const int64_t* mask_ptr, const int32_t* mask_idx, int mode_only_listed, int descending,
                            int32_t n, int32_t* out_ids, float* out_vals, int32_t* out_count, cudaStream_t st) {
  return descending ? rowselect_launch_t<SIGMOID, true>(variant, scores, ld, num_cards, batch, mask_ptr, mask_idx,
                                                        mode_only_listed, n, out_ids, out_vals, out_count, st)
                    : rowselect_launch_t<SIGMOID, false>(variant, scores, ld, num_cards, batch, mask_ptr, mask_idx,
                                                         mode_only_listed, n, out_ids, out_vals, out_count, st);
}

// float32, n <= 128: 0 = automatic (row select when the rows qualify, else the streaming select), 1 = streaming select,
// 2 / 3 = row select with both sweeps over shared memory, one CTA per SM with two row buffers / two CTAs per SM (error
// if the rows do not qualify); 4 = its register form (rows of up to 22 528 cards); automatic takes the register form when
// the row fits and the whole row is ranked, else 3.  The radix-select kernel stays the general path (any n, float64).
static int g_topn_algo = 0;
static int g_topn_force_radix = 0;

template <bool SIGMOID>
static int select_small_n(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                          const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n,
                          int32_t* out_ids, float* out_vals, int32_t* out_count, cudaStream_t st) {
  const bool ok = rowselect_eligible(scores, ld, num_cards, n);
  CC_REQUIRE(ok || g_topn_algo < 2, "cc_topn_masked: the row select needs ld %% 4 == 0, 16-byte aligned rows and C <= ~26 000");
  const bool regs_ok = ((num_cards + 3) >> 2) <= RS_GROUPS * RS_THREADS;
  CC_REQUIRE(regs_ok || g_topn_algo != 4, "cc_topn_masked: the REGS row select holds rows of up to %d cards", 4 * RS_GROUPS * RS_THREADS);
  if (ok && g_topn_algo != 1) {
    // automatic = 2 CTAs per SM; the register form when the row fits its 11 float4 groups per thread and the whole row
    // is ranked (measured 92 us per 4096 cubes against 103 us with both sweeps over shared memory,
    // profiles/r02/topn_bench_regs_v3.jsonl); the only-listed mode never reaches the register path
    const int variant = g_topn_algo == 2 ? 0 : g_topn_algo == 3 ? 1 : (g_topn_algo == 4 || (regs_ok && !mode_only_listed)) ? 2 : 1;
    return rowselect_launch<SIGMOID>(variant, scores, ld, num_cards, batch, mask_ptr, mask_idx,
                                     mode_only_listed, descending, n, out_ids, out_vals, out_count, st);
  }
  return warpselect_launch<SIGMOID>(scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, descending, n,
                                    out_ids, out_vals, out_count, st);
}

// ------------------------------------------------------------------ card similarity
// dist[r] = -cos(emb[r], emb[q]) with Keras' l2_normalize (x * rsqrt(max(sum x^2, 1e-12))), one warp per row
// (reference src/scripts/similarity.py:25-29 evaluates the Keras CosineSimilarity loss once per card in a Python loop)
__global__ void __launch_bounds__(256)
cosine_neg_kernel(const float* __restrict__ emb, int64_t ld, int32_t rows, int32_t dim, int32_t query,
                  float* __restrict__ out) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* a = emb + int64_t(query) * ld;
  const float* b = emb + int64_t(r) * ld;
  float ab = 0.f, aa = 0.f, bb = 0.f;
  for (int k = lane; k < dim; k += 32) {
    const float x = a[k], y = b[k];
    ab = fmaf(x, y, ab); aa = fmaf(x, x, aa); bb = fmaf(y, y, bb);
  }
  ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
  if (lane == 0) out[r] = -(ab * rsqrtf(fmaxf(aa, 1e-12f)) * rsqrtf(fmaxf(bb, 1e-12f)));
}

static int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

template <typename T>
int topn_launch(const T* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n, void* workspace,
                int64_t workspace_bytes, int32_t* out_ids, T* out_vals, int32_t* out_count, cudaStream_t st) {
  using K = typename KeyOf<T>::K;
  CC_REQUIRE(scores && mask_ptr && out_ids, "cc_topn_masked: null pointer");
  CC_REQUIRE(num_cards > 0 && batch >= 0 && n > 0 && ld >= num_cards, "cc_topn_masked: bad sizes");
  if (batch == 0) return CC_OK;
  const size_t mask_bytes = size_t((num_cards + 31) / 32) * 4;
  if constexpr (sizeof(T) == 4) {
    if (n <= WS_MAX_N && !g_topn_force_radix)
      return select_small_n<false>(scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, descending, n,
                                   out_ids, out_vals, out_count, st);
  }
  if (n <= TOPN_MAX_SMEM_N) {
    const int n_pad = next_pow2(n < 2 ? 2 : n);
    const size_t smem = size_t(n_pad) * sizeof(K) + mask_bytes;
    CC_REQUIRE(smem <= 200 * 1024, "cc_topn_masked: C=%d needs %zu bytes of shared memory", num_cards, smem);
    CC_CHECK_CUDA(cudaFuncSetAttribute(topn_masked_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_masked_kernel<T><<<batch, TOPN_THREADS, smem, st>>>(scores, ld, num_cards, mask_ptr, mask_idx,
                                                            mode_only_listed, descending, n, n_pad, out_ids,
                                                            out_vals, out_count);
  } else {
    const int p2 = next_pow2(num_cards);
    const int64_t need = int64_t(batch) * p2 * int64_t(sizeof(K));
    CC_REQUIRE(workspace && workspace_bytes >= need,
               "cc_topn_masked: full ranking needs a %lld-byte workspace (got %lld)", (long long)need,
               (long long)workspace_bytes);
    CC_REQUIRE(mask_bytes <= 200 * 1024, "cc_topn_masked: C too large for the mask");
    CC_CHECK_CUDA(cudaFuncSetAttribute(rank_all_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mask_bytes));
    rank_all_kernel<T><<<batch, 1024, mask_bytes, st>>>(scores, ld, num_cards, mask_ptr, mask_idx, mode_only_listed,
                                                        descending, n, p2, reinterpret_cast<K*>(workspace), out_ids,
                                                        out_vals, out_count);
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// host-side leaf plan of NumPy's pairwise sum over n rows
static void plan_pairwise(int start, int n, int cube, Leaf* out, int* count) {
  if (n <= 128) { out[(*count)++] = Leaf{start, n, 0, cube}; return; }
  int n2 = n / 2; n2 -= n2 % 8;
  plan_pairwise(start, n2, cube, out, count);
  plan_pairwise(start + n2, n - n2, cube, out, count);
  out[*count - 1].merges += 1;
}

}  // namespace cc

using namespace cc;

extern "C" {

int64_t cc_pairwise_leaf_count(int64_t n_rows) {
  if (n_rows <= 128) return 1;
  int64_t n2 = n_rows / 2; n2 -= n2 % 8;
  return cc_pairwise_leaf_count(n2) + cc_pairwise_leaf_count(n_rows - n2);
}

// Builds the leaf plan on the host (plan_host: int32 [total_leaves][4], leaf_ptr_host: int32 [batch+1]).
int cc_pairwise_plan_host(const int64_t* row_ptr_host, int32_t batch, int32_t* plan_host, int32_t* leaf_ptr_host) {
  CC_REQUIRE(row_ptr_host && plan_host && leaf_ptr_host && batch >= 0, "cc_pairwise_plan_host: bad arguments");
  int count = 0;
  leaf_ptr_host[0] = 0;
  for (int b = 0; b < batch; ++b) {
    const int64_t n = row_ptr_host[b + 1] - row_ptr_host[b];
    CC_REQUIRE(n >= 0 && n < (1 << 30), "cc_pairwise_plan_host: bad row count");
    if (n > 0) plan_pairwise(0, (int)n, b, reinterpret_cast<Leaf*>(plan_host), &count);
    leaf_ptr_host[b + 1] = count;
  }
  return CC_OK;
}

int cc_score_gather_f64(const double* m, int64_t ld, int32_t num_cards, const int32_t* rows, const int64_t* row_ptr,
                        int32_t batch, const int32_t* plan, const int32_t* leaf_ptr, int32_t total_leaves,
                        int zero_diag, double* partial_ws, double* scores, int64_t ld_scores, void* stream) {
  CC_NVTX("cc_score_gather_f64");
  CC_REQUIRE(m && rows && row_ptr && plan && leaf_ptr && partial_ws && scores, "cc_score_gather_f64: null pointer");
  CC_REQUIRE(num_cards > 0 && batch >= 0 && ld >= num_cards && ld_scores >= num_cards, "cc_score_gather_f64: bad sizes");
  if (batch == 0) return CC_OK;
  cudaStream_t st = as_stream(stream);
  const int cb = ceil_div(num_cards, 128);
  if (total_leaves > 0) {
    gather_leaf_kernel<<<dim3(cb, total_leaves), 128, 0, st>>>(m, ld, num_cards, rows, row_ptr,
                                                              reinterpret_cast<const Leaf*>(plan), zero_diag, partial_ws);
    CC_CHECK_LAUNCH();
  }
  gather_combine_kernel<<<dim3(cb, batch), 128, 0, st>>>(partial_ws, num_cards, reinterpret_cast<const Leaf*>(plan),
                                                         leaf_ptr, scores, ld_scores);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int64_t cc_topn_workspace_bytes(int32_t num_cards, int32_t batch, int32_t n, int is_f64) {
  if (n <= TOPN_MAX_SMEM_N) return 0;
  return int64_t(batch) * next_pow2(num_cards) * (is_f64 ? 16 : 8);
}

int cc_topn_masked_f32(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                       const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n, void* workspace,
                       int64_t workspace_bytes, int32_t* out_ids, float* out_vals, int32_t* out_count, void* stream) {
  CC_NVTX("cc_topn_masked_f32");
  return topn_launch<float>(scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, descending, n,
                            workspace, workspace_bytes, out_ids, out_vals, out_count, as_stream(stream));
}

// logits in, float32 sigmoid probabilities ranked (ml_recommend.py:78-104): the sigmoid is applied on the fly, so the
// C-wide probability rows are never written.  n <= 128.
int cc_topn_masked_sigmoid_f32(const float* logits, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                               const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n,
                               int32_t* out_ids, float* out_probs, int32_t* out_count, void* stream) {
  CC_NVTX("cc_topn_masked_sigmoid_f32");
  CC_REQUIRE(logits && mask_ptr && out_ids, "cc_topn_masked_sigmoid_f32: null pointer");
  CC_REQUIRE(num_cards > 0 && batch >= 0 && n > 0 && ld >= num_cards, "cc_topn_masked_sigmoid_f32: bad sizes");
  CC_REQUIRE(n <= WS_MAX_N, "cc_topn_masked_sigmoid_f32: n must be <= %d (use cc_sigmoid_f32 + cc_topn_masked_f32)", WS_MAX_N);
  if (batch == 0) return CC_OK;
  return select_small_n<true>(logits, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, descending, n,
                              out_ids, out_probs, out_count, as_stream(stream));
}

int cc_cosine_neg_f32(const float* emb, int64_t ld, int32_t rows, int32_t dim, int32_t query, float* out, void* stream) {
  CC_NVTX("cc_cosine_neg_f32");
  CC_REQUIRE(emb && out && rows > 0 && dim > 0 && ld >= dim && query >= 0 && query < rows, "cc_cosine_neg_f32: bad arguments");
  cosine_neg_kernel<<<ceil_div(rows, 8), 256, 0, as_stream(stream)>>>(emb, ld, rows, dim, query, out);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// 1 = keep float32 top-N on the radix-select kernel even for small n (tests compare the two kernels)
int cc_topn_set_force_radix(int on) { g_topn_force_radix = on ? 1 : 0; return CC_OK; }

// Diagnostic: the fused-sigmoid, descending row select with per-phase clock64() sums of every CTA's thread 0
// (prof: int64 [grid][10] on the device, grid = cc_topn_rowselect_profile_grid(batch, variant); slots: see RS_PROF_SLOTS).
int64_t cc_topn_rowselect_profile_grid(int32_t batch, int variant) {
  const int ctas = variant == 0 ? 1 : 2;
  return batch < ctas * sm_count() ? batch : ctas * sm_count();
}
int cc_topn_rowselect_profile(const float* logits, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                              const int32_t* mask_idx, int32_t n, int variant, int32_t* out_ids, float* out_probs,
                              int32_t* out_count, long long* prof, void* stream) {
  CC_NVTX("cc_topn_rowselect_profile");
  CC_REQUIRE(logits && mask_ptr && out_ids && prof, "cc_topn_rowselect_profile: null pointer");
  CC_REQUIRE(batch > 0 && n > 0 && rowselect_eligible(logits, ld, num_cards, n), "cc_topn_rowselect_profile: rows do not qualify");
  const int nbuf = variant == 0 ? 2 : 1;
  const size_t smem = rowselect_smem_bytes(num_cards, nbuf);
  const int grid = (int)cc_topn_rowselect_profile_grid(batch, variant);
  if (variant == 2) {
    CC_CHECK_CUDA(cudaFuncSetAttribute(topn_rowselect_kernel<true, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_rowselect_kernel<true, true, true, true><<<grid, RS_THREADS, smem, as_stream(stream)>>>(
        logits, ld, num_cards, batch, mask_ptr, mask_idx, 0, n, nbuf, out_ids, out_probs, out_count, prof);
  } else {
    CC_CHECK_CUDA(cudaFuncSetAttribute(topn_rowselect_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_rowselect_kernel<true, true, true><<<grid, RS_THREADS, smem, as_stream(stream)>>>(
        logits, ld, num_cards, batch, mask_ptr, mask_idx, 0, n, nbuf, out_ids, out_probs, out_count, prof);
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// float32 top-N with n <= 128: 0 = automatic, 1 = warp-per-cube streaming select, 2 / 3 = CTA-per-cube row select
// (one CTA per SM with two row buffers / two CTAs per SM with one)
int cc_topn_set_algo(int algo) {
  CC_REQUIRE(algo >= 0 && algo <= 4, "cc_topn_set_algo: algo must be 0..4");
  g_topn_algo = algo;
  return CC_OK;
}

int cc_topn_masked_f64(const double* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                       const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n, void* workspace,
                       int64_t workspace_bytes, int32_t* out_ids, double* out_vals, int32_t* out_count, void* stream) {
  CC_NVTX("cc_topn_masked_f64");
  return topn_launch<double>(scores, ld, num_cards, batch, mask_ptr, mask_idx, mode_only_listed, descending, n,
                             workspace, workspace_bytes, out_ids, out_vals, out_count, as_stream(stream));
}

}  // extern "C"
