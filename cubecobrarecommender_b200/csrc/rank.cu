// Target ranks for leave-k-out evaluation of the recommender: where each held-out card of a cube lands in the list
// the masked top-N select (topn.cu) would return, by the same total order (make_key, cc_common.cuh).
#include "cc_common.cuh"

namespace cc {

// out_rank[p] = #{candidates whose key beats target p's key}: the 0-based slot the descending select would return the
// target at (same make_key order; candidates = cards of [0, C) not listed in the mask row, the targets included).
// One CTA per cube.  The mask row becomes a C-bit bitmap, the targets' keys are sorted ascending in shared memory
// (masked / out-of-range targets get the key RT_NONE and sort past the m real ones), and one sweep over the row does,
// per element, a raw-value compare against the bound of the smallest target key (rs_raw_bound: no element whose key
// beats it is rejected); the few that pass are keyed, binary-searched among the target keys (j = #{target keys < key},
// j >= 1) and counted at cnt[j].  Target i (sorted) is beaten by exactly the elements with j > i: rank[i] =
// sum_{j > i} cnt[j], one block scan.  Equal target keys (duplicate entries) share the first slot's rank: no element
// has its j strictly between them.  A row with more than RT_CHUNK targets takes one sweep per chunk of them.
// T = float (64-bit keys, optional fused sigmoid) or double (96-bit keys in an unsigned __int128, no sigmoid; ld == 0
// is one score row shared by every cube).
constexpr int RT_THREADS = 512;
constexpr int RT_CHUNK = 2 * RT_THREADS;              // target keys per sweep (the scan gives each thread two of them)

// not a candidate: all ones; no real key reaches it (its score word is a NaN)
template <typename K> __device__ __forceinline__ K rt_none() { return ~K(0); }

template <bool SIGMOID> __device__ __forceinline__ float rt_score(float x) { return SIGMOID ? sigmoid_f32(x) : x; }
template <bool SIGMOID> __device__ __forceinline__ double rt_score(double x) { return x; }
template <bool SIGMOID> __device__ __forceinline__ float rt_bound(unsigned long long thr) {
  return rs_raw_bound<SIGMOID>(thr, 1);
}
template <bool SIGMOID> __device__ __forceinline__ double rt_bound(unsigned __int128 thr) {
  return rs_raw_bound_f64(thr, 1);
}

template <typename K>
__device__ __forceinline__ int rt_count_below(const K* keys, int m, K k) {
  int lo = 0, hi = m;                                  // #{i < m : keys[i] < k}, keys ascending
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <typename T, bool SIGMOID>
__global__ void __launch_bounds__(RT_THREADS, 2)
rank_targets_kernel(const T* __restrict__ scores, int64_t ld, int32_t num_cards,
                    const int64_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_idx,
                    const int64_t* __restrict__ target_ptr, const int32_t* __restrict__ target_idx,
                    int32_t* __restrict__ out_rank) {
  static_assert(!SIGMOID || sizeof(T) == 4, "the fused sigmoid ranks float32 logits");
  using K = typename KeyOf<T>::K;
  const K RT_NONE = rt_none<K>();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  K* keys = reinterpret_cast<K*>(smem_raw);                                       // RT_CHUNK, sorted ascending
  int* cnt = reinterpret_cast<int*>(keys + RT_CHUNK);                             // RT_CHUNK + 1 counters, then ranks
  uint32_t* mask = reinterpret_cast<uint32_t*>(cnt + RT_CHUNK + 1);               // ceil(C/32) words
  __shared__ int s_warp[RT_THREADS / 32];
  __shared__ int s_m;
  __shared__ T s_zb;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int cube = blockIdx.x;
  const T* sc = scores + int64_t(cube) * ld;
  const int words = (num_cards + 31) >> 5;
  for (int w = tid; w < words; w += RT_THREADS) mask[w] = 0u;
  __syncthreads();
  for (int64_t p = mask_ptr[cube] + tid; p < mask_ptr[cube + 1]; p += RT_THREADS) {
    const int32_t c = mask_idx[p];
    if (c >= 0 && c < num_cards) atomicOr(&mask[c >> 5], 1u << (c & 31));
  }
  __syncthreads();
  auto target_key = [&](int32_t t) -> K {
    if (t < 0 || t >= num_cards || ((mask[t >> 5] >> (t & 31)) & 1u)) return RT_NONE;
    const T x = sc[t];
    return make_key<T>(rt_score<SIGMOID>(x), (uint32_t)t, 1);
  };
  auto count = [&](T x, int e, T zb) {                 // one candidate element against the chunk's target keys
    if (!(x >= zb) || ((mask[e >> 5] >> (e & 31)) & 1u)) return;
    const K k = make_key<T>(rt_score<SIGMOID>(x), (uint32_t)e, 1);
    const int m = s_m;
    if (k > keys[0]) atomicAdd(&cnt[rt_count_below(keys, m, k)], 1);
  };
  // 16-byte rows: float with ld % 4 == 0, double with ld % 2 == 0 (ld == 0 included), on a 16-byte aligned base
  const bool vec = (ld & (16 / sizeof(T) - 1)) == 0 && (reinterpret_cast<uintptr_t>(scores) & 15) == 0;
  const int64_t tb = target_ptr[cube], te = target_ptr[cube + 1];

  for (int64_t c0 = tb; c0 < te; c0 += RT_CHUNK) {
    const int nt = te - c0 < RT_CHUNK ? (int)(te - c0) : RT_CHUNK;
    int n_pad = 2;
    while (n_pad < nt) n_pad <<= 1;
    for (int i = tid; i < n_pad; i += RT_THREADS) keys[i] = i < nt ? target_key(target_idx[c0 + i]) : RT_NONE;
    for (int i = tid; i <= nt; i += RT_THREADS) cnt[i] = 0;
    __syncthreads();
    for (int k = 2; k <= n_pad; k <<= 1) {             // bitonic sort, ascending
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < n_pad; i += RT_THREADS) {
          const int ixj = i ^ j;
          if (ixj > i) {
            const K a = keys[i], b = keys[ixj];
            if (((i & k) == 0) ? (a > b) : (a < b)) { keys[i] = b; keys[ixj] = a; }
          }
        }
        __syncthreads();
      }
    }
    // m = number of real target keys (they precede the RT_NONE ones)
    if (tid == 0 && keys[0] == RT_NONE) s_m = 0;
    for (int i = tid; i < n_pad; i += RT_THREADS)
      if (keys[i] != RT_NONE && (i + 1 == n_pad || keys[i + 1] == RT_NONE)) s_m = i + 1;
    if (tid == 0 && keys[0] != RT_NONE) s_zb = rt_bound<SIGMOID>(keys[0]);
    __syncthreads();
    const int m = s_m;
    if (m > 0) {
      const T zb = s_zb;
      if constexpr (sizeof(T) == 8) {
        if (vec) {
          // 16-byte loads of whole pairs, two in flight per thread; an odd row's last score is read alone (with
          // ld == 0 the row may end right there)
          const int c2 = num_cards >> 1;
          for (int v = tid; v < c2; v += 2 * RT_THREADS) {
            const int v1 = v + RT_THREADS;
            const double2 q0 = ld_nc_d2(sc + 2 * v);
            const double2 q1 = v1 < c2 ? ld_nc_d2(sc + 2 * v1) : make_double2(-INFINITY, -INFINITY);
            const double2 qs[2] = {q0, q1};
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const double2 q = qs[u];
              const int e0 = 2 * (u ? v1 : v);
              // the sentinel pair past the row is skipped by index: with zb = -inf it would pass the value test
              if ((u && v1 >= c2) || !(fmax(q.x, q.y) >= zb)) continue;
              count(q.x, e0, zb);
              count(q.y, e0 + 1, zb);
            }
          }
          if ((num_cards & 1) && tid == 0) count(sc[num_cards - 1], num_cards - 1, zb);
        } else {
          for (int e = tid; e < num_cards; e += RT_THREADS) count(sc[e], e, zb);
        }
      } else if (vec) {
        // 16-byte loads, two in flight per thread; the float4 past the row's end stays inside ld (ld % 4 == 0)
        const int c4 = (num_cards + 3) >> 2;
        for (int v = tid; v < c4; v += 2 * RT_THREADS) {
          const int v1 = v + RT_THREADS;
          const float4 q0 = ld_nc_f4(sc + 4 * v);
          const float4 q1 = v1 < c4 ? ld_nc_f4(sc + 4 * v1) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
          const float4 qs[2] = {q0, q1};
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const float4 q = qs[u];
            const int e0 = 4 * (u ? v1 : v);
            if (!(fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)) >= zb)) continue;
            const float x[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (e0 + j < num_cards) count(x[j], e0 + j, zb);
          }
        }
      } else {
        for (int e = tid; e < num_cards; e += RT_THREADS) count(sc[e], e, zb);
      }
    }
    __syncthreads();
    // rank[i] = sum_{j > i} cnt[j] for i < m: an inclusive scan of a[q] = cnt[m - q], rank[i] = scan[m - 1 - i]
    {
      const int q0 = 2 * tid, q1 = q0 + 1;
      const int a0 = q0 < m ? cnt[m - q0] : 0, a1 = q1 < m ? cnt[m - q1] : 0;
      int s = a0 + a1;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += y;
      }
      if (lane == 31) s_warp[wid] = s;
      __syncthreads();
      if (wid == 0) {
        int w = lane < RT_THREADS / 32 ? s_warp[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, w, o);
          if (lane >= o) w += y;
        }
        if (lane < RT_THREADS / 32) s_warp[lane] = w;       // inclusive warp totals
      }
      __syncthreads();
      const int before = (wid ? s_warp[wid - 1] : 0) + s - (a0 + a1);
      if (q0 < m) cnt[m - 1 - q0] = before + a0;             // every counter was read above the first barrier
      if (q1 < m) cnt[m - 1 - q1] = before + a0 + a1;
    }
    __syncthreads();
    for (int i = tid; i < nt; i += RT_THREADS) {
      const K k = target_key(target_idx[c0 + i]);
      out_rank[c0 + i] = k == RT_NONE ? -1 : cnt[rt_count_below(keys, m, k)];
    }
    __syncthreads();                                   // keys / cnt are refilled by the next chunk
  }
}

}  // namespace cc

using namespace cc;

extern "C" {

int cc_rank_targets_f32(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                        const int32_t* mask_idx, const int64_t* target_ptr, const int32_t* target_idx, int apply_sigmoid,
                        int32_t* out_rank, void* stream) {
  CC_NVTX("cc_rank_targets_f32");
  CC_REQUIRE(scores && mask_ptr && mask_idx && target_ptr && target_idx && out_rank, "cc_rank_targets_f32: null pointer");
  CC_REQUIRE(num_cards >= 1 && batch >= 0 && ld >= num_cards, "cc_rank_targets_f32: bad sizes (C=%d, batch=%d, ld=%lld)",
             num_cards, batch, (long long)ld);
  if (batch == 0) return CC_OK;
  const size_t smem = size_t(RT_CHUNK) * 8 + size_t(RT_CHUNK + 1) * 4 + size_t((num_cards + 31) / 32) * 4;
  CC_REQUIRE(smem <= 200 * 1024, "cc_rank_targets_f32: C=%d needs %zu bytes of shared memory", num_cards, smem);
  cudaStream_t st = as_stream(stream);
  if (apply_sigmoid) {
    if (smem > 48 * 1024)
      CC_CHECK_CUDA(cudaFuncSetAttribute(rank_targets_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
    rank_targets_kernel<float, true><<<batch, RT_THREADS, smem, st>>>(scores, ld, num_cards, mask_ptr, mask_idx,
                                                                      target_ptr, target_idx, out_rank);
  } else {
    if (smem > 48 * 1024)
      CC_CHECK_CUDA(cudaFuncSetAttribute(rank_targets_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
    rank_targets_kernel<float, false><<<batch, RT_THREADS, smem, st>>>(scores, ld, num_cards, mask_ptr, mask_idx,
                                                                       target_ptr, target_idx, out_rank);
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_rank_targets_f64(const double* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                        const int32_t* mask_idx, const int64_t* target_ptr, const int32_t* target_idx,
                        int32_t* out_rank, void* stream) {
  CC_NVTX("cc_rank_targets_f64");
  CC_REQUIRE(scores && mask_ptr && mask_idx && target_ptr && target_idx && out_rank,
             "cc_rank_targets_f64: null pointer");
  CC_REQUIRE(num_cards >= 1 && batch >= 0 && (ld == 0 || ld >= num_cards),
             "cc_rank_targets_f64: bad sizes (C=%d, batch=%d, ld=%lld)", num_cards, batch, (long long)ld);
  if (batch == 0) return CC_OK;
  const size_t smem = size_t(RT_CHUNK) * 16 + size_t(RT_CHUNK + 1) * 4 + size_t((num_cards + 31) / 32) * 4;
  CC_REQUIRE(smem <= 200 * 1024, "cc_rank_targets_f64: C=%d needs %zu bytes of shared memory", num_cards, smem);
  cudaStream_t st = as_stream(stream);
  if (smem > 48 * 1024)
    CC_CHECK_CUDA(cudaFuncSetAttribute(rank_targets_kernel<double, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
  rank_targets_kernel<double, false><<<batch, RT_THREADS, smem, st>>>(scores, ld, num_cards, mask_ptr, mask_idx,
                                                                      target_ptr, target_idx, out_rank);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

}  // extern "C"
