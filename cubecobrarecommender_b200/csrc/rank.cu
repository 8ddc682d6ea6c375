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
constexpr int RT_THREADS = 512;
constexpr int RT_CHUNK = 2 * RT_THREADS;              // target keys per sweep (the scan gives each thread two of them)
constexpr unsigned long long RT_NONE = ~0ull;         // not a candidate; no real key reaches it (its score word is a NaN)

__device__ __forceinline__ int rt_count_below(const unsigned long long* keys, int m, unsigned long long k) {
  int lo = 0, hi = m;                                  // #{i < m : keys[i] < k}, keys ascending
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <bool SIGMOID>
__global__ void __launch_bounds__(RT_THREADS, 2)
rank_targets_kernel(const float* __restrict__ scores, int64_t ld, int32_t num_cards,
                    const int64_t* __restrict__ mask_ptr, const int32_t* __restrict__ mask_idx,
                    const int64_t* __restrict__ target_ptr, const int32_t* __restrict__ target_idx,
                    int32_t* __restrict__ out_rank) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);     // RT_CHUNK, sorted ascending
  int* cnt = reinterpret_cast<int*>(keys + RT_CHUNK);                             // RT_CHUNK + 1 counters, then ranks
  uint32_t* mask = reinterpret_cast<uint32_t*>(cnt + RT_CHUNK + 1);               // ceil(C/32) words
  __shared__ int s_warp[RT_THREADS / 32];
  __shared__ int s_m;
  __shared__ float s_zb;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int cube = blockIdx.x;
  const float* sc = scores + int64_t(cube) * ld;
  const int words = (num_cards + 31) >> 5;
  for (int w = tid; w < words; w += RT_THREADS) mask[w] = 0u;
  __syncthreads();
  for (int64_t p = mask_ptr[cube] + tid; p < mask_ptr[cube + 1]; p += RT_THREADS) {
    const int32_t c = mask_idx[p];
    if (c >= 0 && c < num_cards) atomicOr(&mask[c >> 5], 1u << (c & 31));
  }
  __syncthreads();
  auto target_key = [&](int32_t t) -> unsigned long long {
    if (t < 0 || t >= num_cards || ((mask[t >> 5] >> (t & 31)) & 1u)) return RT_NONE;
    const float x = sc[t];
    return make_key<float>(SIGMOID ? sigmoid_f32(x) : x, (uint32_t)t, 1);
  };
  auto count = [&](float x, int e, float zb) {         // one candidate element against the chunk's target keys
    if (!(x >= zb) || ((mask[e >> 5] >> (e & 31)) & 1u)) return;
    const unsigned long long k = make_key<float>(SIGMOID ? sigmoid_f32(x) : x, (uint32_t)e, 1);
    const int m = s_m;
    if (k > keys[0]) atomicAdd(&cnt[rt_count_below(keys, m, k)], 1);
  };
  const bool vec = (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(scores) & 15) == 0;
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
            const unsigned long long a = keys[i], b = keys[ixj];
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
    if (tid == 0 && keys[0] != RT_NONE) s_zb = rs_raw_bound<SIGMOID>(keys[0], 1);
    __syncthreads();
    const int m = s_m;
    if (m > 0) {
      const float zb = s_zb;
      if (vec) {
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
      const unsigned long long k = target_key(target_idx[c0 + i]);
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
      CC_CHECK_CUDA(cudaFuncSetAttribute(rank_targets_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rank_targets_kernel<true><<<batch, RT_THREADS, smem, st>>>(scores, ld, num_cards, mask_ptr, mask_idx, target_ptr,
                                                               target_idx, out_rank);
  } else {
    if (smem > 48 * 1024)
      CC_CHECK_CUDA(cudaFuncSetAttribute(rank_targets_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rank_targets_kernel<false><<<batch, RT_THREADS, smem, st>>>(scores, ld, num_cards, mask_ptr, mask_idx, target_ptr,
                                                                target_idx, out_rank);
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

}  // extern "C"
