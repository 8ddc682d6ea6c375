// Losses of the regularised DAE and the optimiser (Keras 2.5 conventions).
//
// Replaces reference src/ml/train.py:83-88:
//   compile(optimizer='adam', loss=['binary_crossentropy','kullback_leibler_divergence'],
//           loss_weights=[1.0, reg])
// * BCE on the sigmoid tower is evaluated from the logits (Keras-2.5 graph path):
//     l = max(z,0) - z*y + log1p(exp(-|z|)),  mean over B*C;  dl/dz = (sigmoid(z)-y)/(B*C)
// * KLD on the softmax tower: t' = clip(t,1e-7,1), q' = clip(softmax(z),1e-7,1),
//     kl = mean_r sum_c t' log(t'/q');  d/dz_c = reg*(q_c*S - t'_c*1[q_c unclipped])/R,
//     S = sum over unclipped c of t'_c
// * Adam: lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v updates; theta -= lr_t*m/(sqrt(v)+eps),
//   eps = 1e-7 outside the bias correction, dense over every parameter.
// These are the unfused forms; gemm_tc.cu carries the BCE math inside the GEMM epilogue.
#include <cuda_bf16.h>

#include "cc_common.cuh"

namespace cc {

constexpr float KERAS_EPS = 1e-7f;

__device__ __forceinline__ double block_sum_double(double v, double* red /* smem[32] */) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  double t = 0.0;
  if (wid == 0) {
    t = lane < (blockDim.x >> 5) ? red[lane] : 0.0;
    t = warp_sum(t);
    if (lane == 0) red[0] = t;
  }
  __syncthreads();
  t = red[0];
  return t;
}
__device__ __forceinline__ float block_max_float(float v, float* red /* smem[32] */) {
  v = warp_max(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float t;
  if (wid == 0) {
    t = lane < (blockDim.x >> 5) ? red[lane] : -INFINITY;
    t = warp_max(t);
    if (lane == 0) red[0] = t;
  }
  __syncthreads();
  t = red[0];
  return t;
}

// ---------------------------------------------------------------- sigmoid-BCE
__global__ void __launch_bounds__(256)
bce_rows_kernel(const float* __restrict__ z, int64_t ldz, const uint32_t* __restrict__ ybits, int64_t ywords,
                int32_t num_cards, int32_t ncols_pad, float inv_count, float* __restrict__ dz, int64_t lddz,
                double* __restrict__ row_loss) {
  __shared__ double red[32];
  const int b = blockIdx.x;
  const float* zr = z + int64_t(b) * ldz;
  const uint32_t* yr = ybits + int64_t(b) * ywords;
  float* dr = dz ? dz + int64_t(b) * lddz : nullptr;
  float s = 0.f;
  for (int c = threadIdx.x; c < ncols_pad; c += blockDim.x) {
    if (c < num_cards) {
      const float v = zr[c];
      const float y = float((yr[c >> 5] >> (c & 31)) & 1u);
      const float e = expf(-fabsf(v));
      s += fmaxf(v, 0.f) - v * y + log1pf(e);
      if (dr) {
        const float sig = v >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
        dr[c] = (sig - y) * inv_count;
      }
    } else if (dr) {
      dr[c] = 0.f;
    }
  }
  const double tot = block_sum_double(double(s), red);
  if (threadIdx.x == 0) row_loss[b] = tot;
}

// Keras binary_accuracy numerator per row: cells with (z > 0) == y  (exact-fp32 mode; the tensor-core modes count
// inside the fused GEMM epilogue)
__global__ void __launch_bounds__(256)
binary_accuracy_rows_kernel(const float* __restrict__ z, int64_t ldz, const uint32_t* __restrict__ ybits, int64_t ywords,
                            int32_t num_cards, double* __restrict__ row_correct) {
  __shared__ double red[32];
  const int b = blockIdx.x;
  const float* zr = z + int64_t(b) * ldz;
  const uint32_t* yr = ybits + int64_t(b) * ywords;
  int hits = 0;
  for (int c = threadIdx.x; c < num_cards; c += blockDim.x)
    hits += ((zr[c] > 0.f) == (((yr[c >> 5] >> (c & 31)) & 1u) != 0u)) ? 1 : 0;
  const double tot = block_sum_double(double(hits), red);
  if (threadIdx.x == 0) row_correct[b] = tot;
}

// ---------------------------------------------------------------- softmax-KL
template <bool CACHE>
__global__ void __launch_bounds__(1024)
softmax_kl_rows_kernel(const float* __restrict__ z, int64_t ldz, const float* __restrict__ target, int64_t ldt,
                       const int32_t* __restrict__ target_rows, int32_t num_cards, int32_t ncols_pad,
                       float grad_scale /* reg / R */, float* __restrict__ dz, int64_t lddz,
                       double* __restrict__ row_loss, int round_tf32) {
  extern __shared__ __align__(16) float srow[];   // CACHE: z row then t row
  __shared__ double redd[32];
  __shared__ float redf[32];
  const int r = blockIdx.x;
  const float* zr = z + int64_t(r) * ldz;
  const float* tr = target + int64_t(target_rows ? target_rows[r] : r) * ldt;
  float* dr = dz ? dz + int64_t(r) * lddz : nullptr;
  float* sz = srow;
  float* stt = srow + num_cards;

  float mx = -INFINITY;
  for (int c = threadIdx.x; c < num_cards; c += blockDim.x) {
    const float v = zr[c];
    if (CACHE) sz[c] = v;
    mx = fmaxf(mx, v);
  }
  mx = block_max_float(mx, redf);
  float se = 0.f;
  for (int c = threadIdx.x; c < num_cards; c += blockDim.x) se += expf((CACHE ? sz[c] : zr[c]) - mx);
  const double sumexp = block_sum_double(double(se), redd);
  const float inv_sum = float(1.0 / sumexp);

  float loss = 0.f, sun = 0.f;
  for (int c = threadIdx.x; c < num_cards; c += blockDim.x) {
    const float q = expf((CACHE ? sz[c] : zr[c]) - mx) * inv_sum;
    const float t = tr[c];
    if (CACHE) stt[c] = t;
    const float tc = fminf(fmaxf(t, KERAS_EPS), 1.f);
    const float qc = fminf(fmaxf(q, KERAS_EPS), 1.f);
    loss += tc * logf(tc / qc);
    if (q >= KERAS_EPS && q <= 1.f) sun += tc;
  }
  const double row = block_sum_double(double(loss), redd);
  const float S = float(block_sum_double(double(sun), redd));
  if (threadIdx.x == 0) row_loss[r] = row;
  if (dr) {
    for (int c = threadIdx.x; c < ncols_pad; c += blockDim.x) {
      float g = 0.f;
      if (c < num_cards) {
        const float q = expf((CACHE ? sz[c] : zr[c]) - mx) * inv_sum;
        const float t = CACHE ? stt[c] : tr[c];
        const float tc = fminf(fmaxf(t, KERAS_EPS), 1.f);
        const bool un = (q >= KERAS_EPS && q <= 1.f);
        g = (q * S - (un ? tc : 0.f)) * grad_scale;
        if (round_tf32) g = rn_tf32(g);
      }
      dr[c] = g;
    }
  }
}


// Fast path (C*4 bytes <= ~100 KB, C % 4 == 0): two 512-thread CTAs per SM, the logits row cached in shared
// memory, 128-bit loads/stores, log q taken from the logits (z - max - lse) instead of a log per element.
//   HBM traffic per row: z read once, target row read once (+ one L2 re-read), dlogits written once.
__device__ __forceinline__ float fast_exp(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f)); return r; }
__device__ __forceinline__ float fast_log(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r * 0.6931471805599453f; }

constexpr int KL_THREADS = 512;

__device__ __forceinline__ float2 block_sum2(float a, float b, float2* red /* smem[16] */) {
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = make_float2(a, b);
  __syncthreads();
  float2 t = lane < (KL_THREADS >> 5) ? red[lane] : make_float2(0.f, 0.f);
  t.x = warp_sum(t.x); t.y = warp_sum(t.y);
  return t;      // every warp reduces the same 16 partials: identical result in all threads
}
__device__ __forceinline__ float block_max1(float a, float2* red) {
  a = warp_max(a);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid].x = a;
  __syncthreads();
  float t = lane < (KL_THREADS >> 5) ? red[lane].x : -INFINITY;
  return warp_max(t);
}

template <bool FAST>   // FAST: MUFU approximations (tensor-core modes); otherwise expf/logf (exact-fp32 mode)
__global__ void __launch_bounds__(KL_THREADS, 2)
softmax_kl_rows_fast_kernel(const float* __restrict__ z, int64_t ldz, const float* __restrict__ target, int64_t ldt,
                            const int32_t* __restrict__ target_rows, int32_t num_cards, int32_t ncols_pad,
                            float grad_scale, float* __restrict__ dz, int64_t lddz, double* __restrict__ row_loss,
                            int round_tf32) {
  auto EXPF = [](float x) { return FAST ? fast_exp(x) : expf(x); };
  auto LOGF = [](float x) { return FAST ? fast_log(x) : logf(x); };
  extern __shared__ __align__(16) float sz[];
  __shared__ float2 red[KL_THREADS / 32];
  const int r = blockIdx.x;
  const float4* z4 = reinterpret_cast<const float4*>(z + int64_t(r) * ldz);
  const float4* t4 = reinterpret_cast<const float4*>(target + int64_t(target_rows ? target_rows[r] : r) * ldt);
  float4* s4 = reinterpret_cast<float4*>(sz);
  const int n4 = num_cards >> 2;

  float mx = -INFINITY;
  for (int i = threadIdx.x; i < n4; i += KL_THREADS) {
    const float4 v = ld_nc_f4(z4 + i);
    s4[i] = v;
    mx = fmaxf(fmaxf(mx, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
  }
  mx = block_max1(mx, red);
  float se = 0.f;
  for (int i = threadIdx.x; i < n4; i += KL_THREADS) {
    const float4 v = s4[i];
    se += (EXPF(v.x - mx) + EXPF(v.y - mx)) + (EXPF(v.z - mx) + EXPF(v.w - mx));
  }
  const float sumexp = block_sum2(se, 0.f, red).x;
  const float inv_sum = 1.f / sumexp;
  const float lse = mx + LOGF(sumexp);
  const float log_eps = -16.11809565095832f;               // log(1e-7)
  float loss = 0.f, sun = 0.f;
  for (int i = threadIdx.x; i < n4; i += KL_THREADS) {
    const float4 v = s4[i];
    const float4 t = __ldg(t4 + i);
    const float zz[4] = {v.x, v.y, v.z, v.w}, tt[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float q = EXPF(zz[k] - mx) * inv_sum;
      const float tc = fminf(fmaxf(tt[k], KERAS_EPS), 1.f);
      const bool un = (q >= KERAS_EPS) && (q <= 1.f);
      const float logq = q >= KERAS_EPS ? fminf(zz[k] - lse, 0.f) : log_eps;   // log(clip(q, 1e-7, 1))
      loss += tc * (LOGF(tc) - logq);
      sun += un ? tc : 0.f;
    }
  }
  const float2 ls = block_sum2(loss, sun, red);
  if (threadIdx.x == 0) row_loss[r] = double(ls.x);
  const float S = ls.y;
  if (dz) {
    float4* d4 = reinterpret_cast<float4*>(dz + int64_t(r) * lddz);
    const int p4 = ncols_pad >> 2;
    for (int i = threadIdx.x; i < p4; i += KL_THREADS) {
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < n4) {
        const float4 v = s4[i];
        const float4 t = __ldg(t4 + i);
        const float zz[4] = {v.x, v.y, v.z, v.w}, tt[4] = {t.x, t.y, t.z, t.w};
        float gg[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float q = EXPF(zz[k] - mx) * inv_sum;
          const float tc = fminf(fmaxf(tt[k], KERAS_EPS), 1.f);
          const bool un = (q >= KERAS_EPS) && (q <= 1.f);
          gg[k] = (q * S - (un ? tc : 0.f)) * grad_scale;
          if (round_tf32) gg[k] = rn_tf32(gg[k]);
        }
        g = make_float4(gg[0], gg[1], gg[2], gg[3]);
      }
      d4[i] = g;
    }
  }
}

// Persistent form with the bias gradient fused in: one 1024-thread CTA per SM walks rows blockIdx.x, + gridDim.x, ...;
// the NEXT row's logits stream into the second half of shared memory (cp.async) while the current row is reduced,
// and every thread keeps the column sums of its dlogits columns in registers across all of the CTA's rows, adding
// them to dbias once at the end (148 x C atomics per launch instead of a separate 344 MB column-sum pass).
constexpr int KLP_THREADS = 1024;
constexpr int KLP_ACC = 7;                 // float4 column accumulators per thread: C <= 4 * 7 * 1024 = 28 672

__device__ __forceinline__ float2 block_sum2_p(float a, float b, float2* red /* smem[32] */) {
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = make_float2(a, b);
  __syncthreads();
  float2 t = red[lane];                    // 32 warps
  t.x = warp_sum(t.x); t.y = warp_sum(t.y);
  return t;
}
__device__ __forceinline__ float block_max1_p(float a, float2* red) {
  a = warp_max(a);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid].x = a;
  __syncthreads();
  return warp_max(red[lane].x);
}

// The row is swept three times out of shared memory: (1) online max / sum of exponentials, (2) loss and S -- here
// exp(z - max) is written back over the logit, so that (3), the gradient sweep, costs no MUFU at all.  With `tlogt`
// (sum_c t'_c log t'_c of every target row, a property of M-hat alone, built once per graph by cc_kl_target_table)
// sweep 2 needs no logarithm either: one ex2 per element in total instead of two ex2 + one lg2 + sweep 1's.
template <bool FAST>
__global__ void __launch_bounds__(KLP_THREADS, 1)
softmax_kl_persistent_kernel(const float* __restrict__ z, int64_t ldz, const float* __restrict__ target, int64_t ldt,
                             const int32_t* __restrict__ target_rows, int32_t rows, int32_t num_cards, int32_t ncols_pad,
                             float grad_scale, float* __restrict__ dz, int64_t lddz, double* __restrict__ row_loss,
                             int round_tf32, float* __restrict__ dbias, __nv_bfloat16* __restrict__ dz16, int64_t lddz16,
                             const double* __restrict__ tlogt, const int32_t* __restrict__ target_argmax,
                             int32_t* __restrict__ row_hit) {
  auto EXPF = [](float x) { return FAST ? fast_exp(x) : expf(x); };
  auto LOGF = [](float x) { return FAST ? fast_log(x) : logf(x); };
  extern __shared__ __align__(16) float sz[];           // two rows of logits
  __shared__ float2 red[KLP_THREADS / 32];
  __shared__ int red_i[KLP_THREADS / 32];
  const int n4 = num_cards >> 2;
  const int p4 = ncols_pad >> 2;
  float4 acc[KLP_ACC];
#pragma unroll
  for (int k = 0; k < KLP_ACC; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);

  auto prefetch = [&](int r, int b) {
    const float4* src = reinterpret_cast<const float4*>(z + int64_t(r) * ldz);
    float4* dst = reinterpret_cast<float4*>(sz) + size_t(b) * n4;
    for (int i = threadIdx.x; i < n4; i += KLP_THREADS) {
      const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(dst + i));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + i) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  int buf = 0;
  int r = blockIdx.x;
  if (r < rows) prefetch(r, 0);
  for (; r < rows; r += gridDim.x) {
    const int rn = r + gridDim.x;
    if (rn < rows) {
      prefetch(rn, buf ^ 1);
      // the next row's TARGET row (a gather out of the 1.7 GB M-hat) is pulled into L2 now, one 128-byte line per thread
      const char* tn = reinterpret_cast<const char*>(target + int64_t(target_rows ? target_rows[rn] : rn) * ldt);
      for (int l = threadIdx.x; l * 128 < num_cards * 4; l += KLP_THREADS)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(tn + size_t(l) * 128));
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    }
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    float4* s4 = reinterpret_cast<float4*>(sz) + size_t(buf) * n4;
    const int64_t trow = target_rows ? target_rows[r] : r;
    const float4* t4 = reinterpret_cast<const float4*>(target + trow * ldt);

    // row maximum and sum of exponentials in ONE sweep and ONE block reduction: every thread keeps (m, s) with
    // s = sum exp(v - m) over its elements, rescaling s when m grows; pairs merge the same way
    float tm = -INFINITY, ts = 0.f;
    for (int i = threadIdx.x; i < n4; i += KLP_THREADS) {
      const float4 v = s4[i];
      const float vm = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
      if (vm > tm) { ts *= EXPF(tm - vm); tm = vm; }
      ts += (EXPF(v.x - tm) + EXPF(v.y - tm)) + (EXPF(v.z - tm) + EXPF(v.w - tm));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, tm, o), os = __shfl_xor_sync(0xffffffffu, ts, o);
      const float nm = fmaxf(tm, om);
      ts = (nm == -INFINITY) ? 0.f : ts * EXPF(tm - nm) + os * EXPF(om - nm);
      tm = nm;
    }
    {
      const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
      __syncthreads();
      if (lane == 0) red[wid] = make_float2(tm, ts);
      __syncthreads();
      float2 t = red[lane];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, t.x, o), os = __shfl_xor_sync(0xffffffffu, t.y, o);
        const float nm = fmaxf(t.x, om);
        t.y = (nm == -INFINITY) ? 0.f : t.y * EXPF(t.x - nm) + os * EXPF(om - nm);
        t.x = nm;
      }
      tm = t.x; ts = t.y;
    }
    const float mx = tm;
    const float sumexp = ts;
    const float inv_sum = 1.f / sumexp;
    const float lse = mx + LOGF(sumexp);
    const float log_eps = -16.11809565095832f;               // log(1e-7)
    // sweep 2: loss = sum t' (log t' - log q'), S = sum of t' over the cards whose q survives the clip; the logit in
    // shared memory is replaced by e = exp(z - max) on the way (each thread rewrites only what it read itself)
    float loss = 0.f, sun = 0.f;
    if (row_hit) {                                          // CTA-uniform: categorical accuracy (see softmax_kl_regs_kernel)
      int cand = 0x7fffffff;
      for (int i = threadIdx.x; i < n4; i += KLP_THREADS) {
        const float4 v = s4[i];
        const int first = v.x == mx ? 0 : v.y == mx ? 1 : v.z == mx ? 2 : v.w == mx ? 3 : -1;
        if (first >= 0) cand = min(cand, 4 * i + first);
      }
      cand = __reduce_min_sync(0xffffffffu, cand);
      __syncthreads();
      if ((threadIdx.x & 31) == 0) red_i[threadIdx.x >> 5] = cand;
      __syncthreads();
      if (threadIdx.x == 0) {
        int best = red_i[0];
        for (int w = 1; w < KLP_THREADS / 32; ++w) best = min(best, red_i[w]);
        row_hit[r] = (best == target_argmax[trow]) ? 1 : 0;
      }
    }
    for (int i = threadIdx.x; i < n4; i += KLP_THREADS) {
      const float4 v = s4[i];
      const float4 t = __ldg(t4 + i);
      const float zz[4] = {v.x, v.y, v.z, v.w}, tt[4] = {t.x, t.y, t.z, t.w};
      float ee[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        ee[k] = EXPF(zz[k] - mx);
        const float q = ee[k] * inv_sum;
        const float tc = fminf(fmaxf(tt[k], KERAS_EPS), 1.f);
        const bool un = (q >= KERAS_EPS) && (q <= 1.f);
        const float logq = q >= KERAS_EPS ? fminf(zz[k] - lse, 0.f) : log_eps;   // log(clip(q, 1e-7, 1))
        if (tlogt) loss -= tc * logq;
        else loss += tc * (LOGF(tc) - logq);
        sun += un ? tc : 0.f;
      }
      s4[i] = make_float4(ee[0], ee[1], ee[2], ee[3]);
    }
    const float2 ls = block_sum2_p(loss, sun, red);
    if (threadIdx.x == 0) row_loss[r] = tlogt ? tlogt[trow] + double(ls.x) : double(ls.x);
    const float S = ls.y;
    const float qs = inv_sum * S * grad_scale;            // dz = (q S - t' 1[unclipped]) scale = e (S scale / sum) - ...
    float4* d4 = dz16 ? nullptr : reinterpret_cast<float4*>(dz + int64_t(r) * lddz);
    uint2* d16 = dz16 ? reinterpret_cast<uint2*>(dz16 + int64_t(r) * lddz16) : nullptr;   // bf16 dlogits ("bf16" mode)
#pragma unroll
    for (int k = 0; k < KLP_ACC + 1; ++k) {
      const int i = threadIdx.x + k * KLP_THREADS;
      if (i >= p4) break;
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < n4) {
        const float4 v = s4[i];                             // e = exp(z - max), left there by sweep 2
        const float4 t = __ldg(t4 + i);
        const float ev[4] = {v.x, v.y, v.z, v.w}, tt[4] = {t.x, t.y, t.z, t.w};
        float gg[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float q = ev[e] * inv_sum;
          const float tc = fminf(fmaxf(tt[e], KERAS_EPS), 1.f);
          const bool un = (q >= KERAS_EPS) && (q <= 1.f);
          gg[e] = FAST ? fmaf(ev[e], qs, un ? -tc * grad_scale : 0.f) : (q * S - (un ? tc : 0.f)) * grad_scale;
          if (round_tf32) gg[e] = rn_tf32(gg[e]);
        }
        g = make_float4(gg[0], gg[1], gg[2], gg[3]);
        if (k < KLP_ACC) { acc[k].x += g.x; acc[k].y += g.y; acc[k].z += g.z; acc[k].w += g.w; }
      }
      if (d16) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(g.x, g.y), hi = __floats2bfloat162_rn(g.z, g.w);
        d16[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
      } else {
        d4[i] = g;
      }
    }
    __syncthreads();          // every thread is done with sz[buf] before the prefetch after next overwrites it
    buf ^= 1;
  }
  if (dbias) {
#pragma unroll
    for (int k = 0; k < KLP_ACC; ++k) {
      const int i = threadIdx.x + k * KLP_THREADS;
      if (i < n4) {
        atomicAdd(dbias + 4 * i, acc[k].x); atomicAdd(dbias + 4 * i + 1, acc[k].y);
        atomicAdd(dbias + 4 * i + 2, acc[k].z); atomicAdd(dbias + 4 * i + 3, acc[k].w);
      }
    }
  }
}

// Register-resident form (the shipped one for C <= 22 528 cards).  The 1024-thread kernel
// above has ONE 16-byte target load in flight per thread (16 KB per SM) and re-reads the target row in its third sweep:
// it is bound by load latency, not by HBM or by the MUFU pipe (measured 0.30 ms for 1.03 GB = 52% of the HBM peak, and
// unchanged when three of its four MUFU ops per element were removed).  Here a CTA has 512-768 threads with 85-128
// registers each: a thread issues ALL of its target loads for the row (7-11 x 16 bytes, 84-88 KB in flight per SM) before
// the first sweep, keeps them in registers for sweeps 2 and 3, and keeps the bias-gradient column sums in registers
// across rows as before.  The logits row still arrives by cp.async one row ahead, the next target row is prefetched
// into L2.
// Two launch shapes, chosen by the row length: 768 threads x 7 slots (85 registers per thread, 24 warps: rows of up to
// 21 504 cards -- the 20 884 of the shipped checkpoints) and 512 threads x 11 slots (128 registers, 16 warps: up to 22 528).
// More warps hide more of the shared-memory / MUFU latencies the kernel stalls on (ncu: profiles/r02/kl_regs_v1_stalls.txt).
// GRAD = false (evaluation, cc_softmax_kl_loss): the kernel stops after sweep 2 -- row_loss / row_hit as with GRAD, no
// dlogits, no column sums, nothing written back to shared memory; 8 bytes per element instead of 12.
template <int WARPS>
__device__ __forceinline__ float2 block_sum2_r(float a, float b, float2* red /* smem[WARPS] */) {
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = make_float2(a, b);
  __syncthreads();
  float2 t = lane < WARPS ? red[lane] : make_float2(0.f, 0.f);      // every warp reduces the same partials
  t.x = warp_sum(t.x); t.y = warp_sum(t.y);
  return t;
}

template <bool FAST, int KLR_THREADS, int ITERS, bool GRAD = true>
__global__ void __launch_bounds__(KLR_THREADS, 1)
softmax_kl_regs_kernel(const float* __restrict__ z, int64_t ldz, const float* __restrict__ target, int64_t ldt,
                       const int32_t* __restrict__ target_rows, int32_t rows, int32_t num_cards, int32_t ncols_pad,
                       float grad_scale, float* __restrict__ dz, int64_t lddz, double* __restrict__ row_loss,
                       int round_tf32, float* __restrict__ dbias, __nv_bfloat16* __restrict__ dz16, int64_t lddz16,
                       const double* __restrict__ tlogt, const int32_t* __restrict__ target_argmax,
                       int32_t* __restrict__ row_hit) {
  // lets the dependent tcgen05 GEMM (programmatic stream serialisation) be scheduled and run its prologue while this grid
  // drains; it still waits (griddepcontrol.wait) for this grid's completion before touching memory
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  auto EXPF = [](float x) { return FAST ? fast_exp(x) : expf(x); };
  auto LOGF = [](float x) { return FAST ? fast_log(x) : logf(x); };
  extern __shared__ __align__(16) float sz[];           // two rows of logits
  __shared__ float2 red[KLR_THREADS / 32];
  __shared__ int red_i[KLR_THREADS / 32];
  const int n4 = num_cards >> 2;
  const int p4 = ncols_pad >> 2;
  float4 acc[ITERS];
#pragma unroll
  for (int k = 0; k < ITERS; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);

  auto prefetch = [&](int r, int b) {
    const float4* src = reinterpret_cast<const float4*>(z + int64_t(r) * ldz);
    float4* dst = reinterpret_cast<float4*>(sz) + size_t(b) * n4;
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      if (i < n4) {
        const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(dst + i));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + i) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  int buf = 0;
  int r = blockIdx.x;
  if (r < rows) prefetch(r, 0);
  for (; r < rows; r += gridDim.x) {
    const int64_t trow = target_rows ? target_rows[r] : r;
    const float4* t4 = reinterpret_cast<const float4*>(target + trow * ldt);
    // this row's targets: every load is issued now and lands while the logits are reduced
    float4 tv[ITERS];
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      tv[k] = i < n4 ? ld_nc_f4(t4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int rn = r + gridDim.x;
    if (rn < rows) {
      prefetch(rn, buf ^ 1);
      const char* tn = reinterpret_cast<const char*>(target + int64_t(target_rows ? target_rows[rn] : rn) * ldt);
      for (int l = threadIdx.x; l * 128 < num_cards * 4; l += KLR_THREADS)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(tn + size_t(l) * 128));
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    float4* s4 = reinterpret_cast<float4*>(sz) + size_t(buf) * n4;

    // sweep 1: row maximum, then the sum of exponentials
    float tm = -INFINITY;
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      if (i < n4) {
        const float4 v = s4[i];
        tm = fmaxf(tm, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
      }
    }
    tm = warp_max(tm);
    {
      const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
      if (lane == 0) red[wid].x = tm;
      __syncthreads();
      tm = warp_max(lane < KLR_THREADS / 32 ? red[lane].x : -INFINITY);
    }
    const float mx = tm;
    // exp(z - max): FAST folds the subtraction into the exponent's scaling, ex2(z * log2e - max * log2e): one FFMA + MUFU
    const float mxl = mx * 1.4426950408889634f;
    auto EXPM = [&](float zc) -> float {
      if (FAST) { float e; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fmaf(zc, 1.4426950408889634f, -mxl))); return e; }
      return expf(zc - mx);
    };
    float ts = 0.f;
    int cand = 0x7fffffff;                                  // first column holding the row maximum (metrics only)
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      if (i < n4) {
        const float4 v = s4[i];
        ts += (EXPM(v.x) + EXPM(v.y)) + (EXPM(v.z) + EXPM(v.w));
        if (row_hit) {                                      // CTA-uniform
          const int first = v.x == mx ? 0 : v.y == mx ? 1 : v.z == mx ? 2 : v.w == mx ? 3 : -1;
          if (first >= 0) cand = min(cand, 4 * i + first);
        }
      }
    }
    const float sumexp = block_sum2_r<KLR_THREADS / 32>(ts, 0.f, red).x;
    if (row_hit) {
      // Keras categorical_accuracy (metrics=['accuracy'] on the softmax output): argmax of the prediction (first maximal
      // column, like tf.argmax) against the argmax of the target row, a per-row table
      cand = __reduce_min_sync(0xffffffffu, cand);
      if ((threadIdx.x & 31) == 0) red_i[threadIdx.x >> 5] = cand;
      __syncthreads();
      if (threadIdx.x == 0) {
        int best = red_i[0];
#pragma unroll
        for (int w = 1; w < KLR_THREADS / 32; ++w) best = min(best, red_i[w]);
        row_hit[r] = (best == target_argmax[trow]) ? 1 : 0;
      }
    }
    const float inv_sum = 1.f / sumexp;
    const float lse = mx + LOGF(sumexp);
    const float log_eps = -16.11809565095832f;               // log(1e-7)
    // q = e / sumexp is clipped to [1e-7, 1] by Keras.  q <= 1 holds by construction (every e <= 1 and the maximum
    // contributes exp(0) = 1 to the sum), so the clip acts iff e < 1e-7 * sumexp: one compare against a row constant
    const float e_clip = KERAS_EPS * sumexp;
    // sweep 2: loss = sum t' (log t' - log q'), S = sum of t' over the cards whose q survives the clip.  The logit is
    // needed one last time here (log q = z - lse); e = exp(z - max) replaces it in shared memory for sweep 3 (keeping
    // both z and e in registers across the reduction would not fit beside the targets and the column sums), and the
    // clipped target t' replaces the raw one in the registers
    float loss = 0.f, sun = 0.f;
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      if (i < n4) {
        const float4 v = s4[i];
        const float zz[4] = {v.x, v.y, v.z, v.w};
        float tt[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
        float ee[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          ee[c] = EXPM(zz[c]);
          tt[c] = fminf(fmaxf(tt[c], KERAS_EPS), 1.f);
          const bool un = ee[c] >= e_clip;
          const float zl = FAST ? zz[c] - lse : fminf(zz[c] - lse, 0.f);
          const float logq = un ? zl : log_eps;             // log(clip(q, 1e-7, 1))
          if (tlogt) loss = fmaf(-tt[c], logq, loss);
          else loss += tt[c] * (LOGF(tt[c]) - logq);
          sun += un ? tt[c] : 0.f;
        }
        if constexpr (GRAD) {
          s4[i] = make_float4(ee[0], ee[1], ee[2], ee[3]);
          tv[k] = make_float4(tt[0], tt[1], tt[2], tt[3]);
        }
      }
    }
    const float2 ls = block_sum2_r<KLR_THREADS / 32>(loss, GRAD ? sun : 0.f, red);
    if (threadIdx.x == 0) row_loss[r] = tlogt ? tlogt[trow] + double(ls.x) : double(ls.x);
    if constexpr (!GRAD) {
      __syncthreads();        // every thread is done with sz[buf] before the prefetch after next overwrites it
      buf ^= 1;
      continue;
    }
    const float S = ls.y;
    const float qs = inv_sum * S * grad_scale;
    float4* d4 = dz16 ? nullptr : reinterpret_cast<float4*>(dz + int64_t(r) * lddz);
    uint2* d16 = dz16 ? reinterpret_cast<uint2*>(dz16 + int64_t(r) * lddz16) : nullptr;
    // sweep 3: dlogits = (q S - t' 1[unclipped]) scale = e (S scale / sumexp) - (t' scale) 1[unclipped]; column sums; store
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      if (i < p4) {
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n4) {
          const float4 e4 = s4[i];
          const float ev[4] = {e4.x, e4.y, e4.z, e4.w}, tt[4] = {tv[k].x, tv[k].y, tv[k].z, tv[k].w};
          float gg[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const bool un = ev[c] >= e_clip;
            gg[c] = FAST ? fmaf(ev[c], qs, un ? -tt[c] * grad_scale : 0.f)
                         : (ev[c] * inv_sum * S - (un ? tt[c] : 0.f)) * grad_scale;
            if (round_tf32) gg[c] = rn_tf32_bits(gg[c]);
          }
          g = make_float4(gg[0], gg[1], gg[2], gg[3]);
          acc[k].x += g.x; acc[k].y += g.y; acc[k].z += g.z; acc[k].w += g.w;
        }
        if (d16) {
          const __nv_bfloat162 lo = __floats2bfloat162_rn(g.x, g.y), hi = __floats2bfloat162_rn(g.z, g.w);
          d16[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
        } else {
          d4[i] = g;
        }
      }
    }
    // pad columns beyond the last register slot (ncols_pad - num_cards < 128 columns: one more slot at most)
    {
      const int i = threadIdx.x + ITERS * KLR_THREADS;
      if (i < p4) {
        if (d16) d16[i] = make_uint2(0u, 0u); else d4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    __syncthreads();          // every thread is done with sz[buf] before the prefetch after next overwrites it
    buf ^= 1;
  }
  if (GRAD && dbias) {
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = threadIdx.x + k * KLR_THREADS;
      if (i < n4) {
        atomicAdd(dbias + 4 * i, acc[k].x); atomicAdd(dbias + 4 * i + 1, acc[k].y);
        atomicAdd(dbias + 4 * i + 2, acc[k].z); atomicAdd(dbias + 4 * i + 3, acc[k].w);
      }
    }
  }
}

// sum_c t'_c log t'_c, t' = clip(t, 1e-7, 1), of every row of the target matrix (M-hat), in float64: the part of the
// Keras KLD that does not depend on the model.  One CTA per row; built once per graph.
__global__ void __launch_bounds__(256)
kl_target_table_kernel(const float* __restrict__ target, int64_t ldt, int32_t num_cards, double* __restrict__ out) {
  __shared__ double red[32];
  const float* tr = target + int64_t(blockIdx.x) * ldt;
  double s = 0.0;
  for (int c = threadIdx.x; c < num_cards; c += blockDim.x) {
    const double tc = double(fminf(fmaxf(tr[c], KERAS_EPS), 1.f));
    s += tc * log(tc);
  }
  s = block_sum_double(s, red);
  if (threadIdx.x == 0) out[blockIdx.x] = s;
}

// loss[0] = bce mean, loss[1] = kl mean, loss[2] = bce + reg*kl   (fixed summation order)
__global__ void __launch_bounds__(1024)
loss_finalize_kernel(const double* __restrict__ bce_rows, int nb, double bce_div, const double* __restrict__ kl_rows,
                     int nr, double kl_div, double reg, double* __restrict__ out) {
  __shared__ double red[32];
  double a = 0.0, k = 0.0;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) a += bce_rows[i];
  for (int i = threadIdx.x; i < nr; i += blockDim.x) k += kl_rows[i];
  a = block_sum_double(a, red);
  k = block_sum_double(k, red);
  if (threadIdx.x == 0) {
    const double bce = bce_div > 0 ? a / bce_div : 0.0, kl = kl_div > 0 ? k / kl_div : 0.0;
    out[0] = bce; out[1] = kl; out[2] = bce + reg * kl;
  }
}

// ------------------------------------------------------------------- Adam
// One definition with explicit rounding steps (no compiler-chosen FMA contraction), so the plain kernel and the
// peer-memory kernel produce identical bits from identical inputs.
__device__ __forceinline__ void adam_update(float& p, float g, float& m, float& v, float b1, float b2, float lr_t,
                                            float eps) {
  m = __fmaf_rn(b1, m, __fmul_rn(1.f - b1, g));
  v = __fmaf_rn(b2, v, __fmul_rn(__fmul_rn(1.f - b2, g), g));
  p = __fsub_rn(p, __fdiv_rn(__fmul_rn(lr_t, m), __fadd_rn(__fsqrt_rn(v), eps)));
}
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
            int64_t n, const int64_t* __restrict__ step_ptr, float lr, float b1, float b2, float eps,
            float* __restrict__ shadow_tf32) {
  const double t = double(*step_ptr + 1);
  const float lr_t = float(double(lr) * sqrt(1.0 - pow(double(b2), t)) / (1.0 - pow(double(b1), t)));
  const int64_t i4 = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i4 + 3 < n) {
    float4 pv = *reinterpret_cast<float4*>(p + i4);
    const float4 gv = *reinterpret_cast<const float4*>(g + i4);
    float4 mv = *reinterpret_cast<float4*>(m + i4);
    float4 vv = *reinterpret_cast<float4*>(v + i4);
    adam_update(pv.x, gv.x, mv.x, vv.x, b1, b2, lr_t, eps);
    adam_update(pv.y, gv.y, mv.y, vv.y, b1, b2, lr_t, eps);
    adam_update(pv.z, gv.z, mv.z, vv.z, b1, b2, lr_t, eps);
    adam_update(pv.w, gv.w, mv.w, vv.w, b1, b2, lr_t, eps);
    *reinterpret_cast<float4*>(p + i4) = pv;
    if (shadow_tf32) {   // tf32 (round-to-nearest) copy of the weights for the tensor-core GEMMs
      float4 sv = pv;
      sv.x = rn_tf32(sv.x); sv.y = rn_tf32(sv.y);
      sv.z = rn_tf32(sv.z); sv.w = rn_tf32(sv.w);
      *reinterpret_cast<float4*>(shadow_tf32 + i4) = sv;
    }
    *reinterpret_cast<float4*>(m + i4) = mv;
    *reinterpret_cast<float4*>(v + i4) = vv;
  } else {
    for (int64_t i = i4; i < n; ++i) {
      float pi = p[i], mi = m[i], vi = v[i];
      adam_update(pi, g[i], mi, vi, b1, b2, lr_t, eps);
      m[i] = mi; v[i] = vi;
      p[i] = pi;
      if (shadow_tf32) { float sv = pi; sv = rn_tf32(sv); shadow_tf32[i] = sv; }
    }
  }
}

// ---------------------------------------------- Adam fused with the gradient exchange over NVLink peer memory
// Data-parallel step, one kernel per rank instead of  all_reduce(grads) -> Adam(all parameters)  on every rank:
// rank r owns the slice [lo, hi) of the flat parameter buffer.  For its slice it
//   (1) loads the gradient from EVERY rank's gradient buffer (local load + peer loads through NVLink / NVSwitch)
//       and sums them in rank order                                                   -> reduce-scatter
//   (2) applies the TF-style Adam update to its slice of m, v, params (1/world of the work and of the HBM traffic)
//   (3) stores the updated parameters into EVERY rank's parameter buffer (peer stores) -> all-gather
// so the collective's transfers ride inside the optimiser pass.  The buffers live in symmetric memory
// (torch.distributed._symmetric_memory); the caller brackets the kernel with two cross-rank barriers
// (all gradients complete before, all parameter slices landed after).
constexpr int P2P_MAX_WORLD = 16;
struct PeerPtrs {
  const float* grads[P2P_MAX_WORLD];
  float* params[P2P_MAX_WORLD];
  const float* grads_mc;          // multicast (NVLS) views of the same buffers, or null
  float* params_mc;
};

__device__ __forceinline__ float4 multimem_ld_reduce_add_f4(const float* mc) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
  return r;
}
__device__ __forceinline__ void multimem_st_f4(float* mc, const float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
               ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// WORLD_CAP: compile-time bound of the rank loops (2, 4, 8, 16) so the per-rank partials stay in registers.
// MULTICAST: the reduction and the broadcast are done by the NVSwitch (multimem.ld_reduce / multimem.st on the
// multicast mapping): one load returns the sum over all ranks, one store reaches all ranks -- NVLink traffic per
// GPU drops from 2 * (world-1)/world to (world+1)/world... of the buffer in the binding direction.
template <int WORLD_CAP, bool MULTICAST>
__global__ void __launch_bounds__(256)
adam_p2p_kernel(const PeerPtrs pp, int world, int rank, float* __restrict__ m, float* __restrict__ v, int64_t lo,
                int64_t hi, const int64_t* __restrict__ step_ptr, float lr, float b1, float b2, float eps) {
  const double t = double(*step_ptr + 1);
  const float lr_t = float(double(lr) * sqrt(1.0 - pow(double(b2), t)) / (1.0 - pow(double(b1), t)));
  // U float4 per thread, one CTA-width apart (coalesced), every remote access of all U issued before the first use:
  // the NVLink round trip is ~2-4 us, so bytes in flight per SM decide the bandwidth
  constexpr int U = MULTICAST ? 4 : (WORLD_CAP <= 4 ? 2 : 1);
  const int64_t base = lo + (int64_t(blockIdx.x) * blockDim.x * U + threadIdx.x) * 4;
  float4 gv[U];
  bool live[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t i4 = base + int64_t(u) * blockDim.x * 4;
    live[u] = i4 < hi;                                     // lo, hi are multiples of 4
    gv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (MULTICAST) {
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (live[u]) gv[u] = multimem_ld_reduce_add_f4(pp.grads_mc + base + int64_t(u) * blockDim.x * 4);   // summed in the switch
  } else {
    float4 part[U][WORLD_CAP];
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int r = 0; r < WORLD_CAP; ++r)
        if (r < world && live[u]) part[u][r] = ld_nc_f4(pp.grads[r] + base + int64_t(u) * blockDim.x * 4);
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int r = 0; r < WORLD_CAP; ++r)                  // fixed rank order: every rank would compute the same sum
        if (r < world && live[u]) {
          gv[u].x += part[u][r].x; gv[u].y += part[u][r].y; gv[u].z += part[u][r].z; gv[u].w += part[u][r].w;
        }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (!live[u]) continue;
    const int64_t i4 = base + int64_t(u) * blockDim.x * 4;
    float4 pv = *reinterpret_cast<const float4*>(pp.params[rank] + i4);
    float4 mv = *reinterpret_cast<float4*>(m + i4);
    float4 vv = *reinterpret_cast<float4*>(v + i4);
    const float4 g = gv[u];
    adam_update(pv.x, g.x, mv.x, vv.x, b1, b2, lr_t, eps);
    adam_update(pv.y, g.y, mv.y, vv.y, b1, b2, lr_t, eps);
    adam_update(pv.z, g.z, mv.z, vv.z, b1, b2, lr_t, eps);
    adam_update(pv.w, g.w, mv.w, vv.w, b1, b2, lr_t, eps);
    *reinterpret_cast<float4*>(m + i4) = mv;
    *reinterpret_cast<float4*>(v + i4) = vv;
    if (MULTICAST) {
      multimem_st_f4(pp.params_mc + i4, pv);               // one store, replicated to every rank by the switch
    } else {
#pragma unroll
      for (int r = 0; r < WORLD_CAP; ++r)
        if (r < world) *reinterpret_cast<float4*>(pp.params[r] + i4) = pv;
    }
  }
  // no per-thread system fence (it serialised every warp on the NVLink round trip: 0.50 -> 0.21 ms at 2 GPUs): grid
  // completion makes the peer stores visible, and the caller's cross-rank barrier only starts after it
}

// fp32 [rows][ld_src] -> bf16 [rows][ld_dst] (round to nearest even), 4 elements per thread; columns in
// [cols, ld_dst) are left untouched
__global__ void convert_f32_bf16_kernel(const float* __restrict__ src, int64_t ld_src, __nv_bfloat16* __restrict__ dst,
                                        int64_t ld_dst, int rows, int cols4) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= int64_t(rows) * cols4) return;
  const int r = int(i / cols4), c4 = int(i % cols4);
  const float4 v = *reinterpret_cast<const float4*>(src + int64_t(r) * ld_src + 4 * c4);
  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  *reinterpret_cast<uint2*>(dst + int64_t(r) * ld_dst + 4 * c4) =
      make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}

__global__ void round_tf32_kernel(const float* __restrict__ x, float* __restrict__ out, int64_t n) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) { float v = x[i]; v = rn_tf32(v); out[i] = v; }
}

// sigmoid of the winners / in-cube scores: probs = 1/(1+exp(-z))
__global__ void sigmoid_kernel(const float* __restrict__ z, float* __restrict__ out, int64_t n) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = sigmoid_f32(z[i]);
}

}  // namespace cc

using namespace cc;

// 0 = choose (the register-resident kernel when the row fits: 768 threads x 7 slots, else 512 x 11), 1 = always the
// 1024-thread kernel, 2 = the register-resident kernel in its 512-thread shape only (cc_softmax_kl_set_variant; tests
// and A/B measurements)
static int g_kl_variant = 0;

extern "C" {

int cc_softmax_kl_set_variant(int variant) {
  CC_REQUIRE(variant >= 0 && variant <= 2, "cc_softmax_kl_set_variant: 0 (auto), 1 (1024-thread kernel) or 2 (512-thread register kernel)");
  g_kl_variant = variant;
  return CC_OK;
}

int cc_bce_logits_fwd_bwd(const float* z, int64_t ldz, const uint32_t* ybits, int64_t ywords, int32_t batch,
                          int32_t num_cards, int32_t ncols_pad, double count /* global B*C */, float* dz,
                          int64_t lddz, double* row_loss, void* stream) {
  CC_NVTX("cc_bce_logits_fwd_bwd");
  CC_REQUIRE(z && ybits && row_loss, "cc_bce_logits_fwd_bwd: null pointer");
  CC_REQUIRE(num_cards > 0 && ncols_pad >= num_cards && ywords * 32 >= num_cards && count > 0,
             "cc_bce_logits_fwd_bwd: bad sizes");
  CC_REQUIRE(!dz || lddz >= ncols_pad, "cc_bce_logits_fwd_bwd: lddz too small");
  if (batch == 0) return CC_OK;
  bce_rows_kernel<<<batch, 256, 0, as_stream(stream)>>>(z, ldz, ybits, ywords, num_cards, ncols_pad,
                                                       float(1.0 / count), dz, lddz, row_loss);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_binary_accuracy_rows(const float* z, int64_t ldz, const uint32_t* ybits, int64_t ywords, int32_t batch,
                            int32_t num_cards, double* row_correct, void* stream) {
  CC_NVTX("cc_binary_accuracy_rows");
  CC_REQUIRE(z && ybits && row_correct && num_cards > 0 && ywords * 32 >= num_cards, "cc_binary_accuracy_rows: bad arguments");
  if (batch == 0) return CC_OK;
  binary_accuracy_rows_kernel<<<batch, 256, 0, as_stream(stream)>>>(z, ldz, ybits, ywords, num_cards, row_correct);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// dbias (nullable, float [num_cards]): receives the column sums of dz (= the softmax layer's bias gradient).  Fused into
// the persistent kernel when it applies (float atomics: last bits vary between runs); otherwise the caller still has
// cc_colsum_f32 -- the return value of cc_softmax_kl_fuses_dbias tells which.
int cc_softmax_kl_fuses_dbias(int32_t num_cards, int32_t ncols_pad, int64_t ldz, int64_t ldt, int64_t lddz) {
  return (num_cards % 4 == 0) && (ldz % 4 == 0) && (ldt % 4 == 0) && (ncols_pad % 4 == 0) && (lddz % 4 == 0) &&
         size_t(num_cards) * 8 <= 200 * 1024 && (ncols_pad >> 2) <= (KLP_ACC + 1) * KLP_THREADS &&
         (num_cards >> 2) <= KLP_ACC * KLP_THREADS;
}

int cc_softmax_kl_fwd_bwd(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                          int32_t rows, int32_t num_cards, int32_t ncols_pad, double grad_scale, float* dz,
                          int64_t lddz, double* row_loss, int round_tf32, float* dbias, void* stream) {
  CC_NVTX("cc_softmax_kl_fwd_bwd");
  return cc_softmax_kl_fwd_bwd_ex(z, ldz, target, ldt, target_rows, rows, num_cards, ncols_pad, grad_scale, dz, lddz, row_loss,
                                  round_tf32, dbias, nullptr, 0, nullptr, stream);
}

int cc_kl_target_table(const float* target, int64_t ldt, int32_t target_rows, int32_t num_cards, double* tlogt, void* stream) {
  CC_NVTX("cc_kl_target_table");
  CC_REQUIRE(target && tlogt && target_rows >= 0 && num_cards > 0 && ldt >= num_cards, "cc_kl_target_table: bad arguments");
  if (target_rows == 0) return CC_OK;
  kl_target_table_kernel<<<target_rows, 256, 0, as_stream(stream)>>>(target, ldt, num_cards, tlogt);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_softmax_kl_fwd_bwd_ex(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                             int32_t rows, int32_t num_cards, int32_t ncols_pad, double grad_scale, float* dz,
                             int64_t lddz, double* row_loss, int round_tf32, float* dbias, void* dz_bf16, int64_t lddz_bf16,
                             const double* tlogt, void* stream) {
  return cc_softmax_kl_fwd_bwd_metrics(z, ldz, target, ldt, target_rows, rows, num_cards, ncols_pad, grad_scale, dz, lddz,
                                       row_loss, round_tf32, dbias, dz_bf16, lddz_bf16, tlogt, nullptr, nullptr, stream);
}

// target_argmax[i] = first maximal column of target row i (int32, one entry per row of the target matrix).
__global__ void __launch_bounds__(256)
kl_target_argmax_kernel(const float* __restrict__ target, int64_t ldt, int32_t num_cards, int32_t* __restrict__ out) {
  __shared__ float redv[8];
  __shared__ int redi[8];
  const float* tr = target + int64_t(blockIdx.x) * ldt;
  float bv = -INFINITY; int bi = 0x7fffffff;
  for (int c = threadIdx.x; c < num_cards; c += blockDim.x) {
    const float v = tr[c];
    if (v > bv) { bv = v; bi = c; }                       // strict: a thread's columns ascend, the first maximum stays
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if ((threadIdx.x & 31) == 0) { redv[threadIdx.x >> 5] = bv; redi[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) if (redv[w] > bv || (redv[w] == bv && redi[w] < bi)) { bv = redv[w]; bi = redi[w]; }
    out[blockIdx.x] = bi;
  }
}

int cc_kl_target_argmax(const float* target, int64_t ldt, int32_t target_rows, int32_t num_cards, int32_t* out, void* stream) {
  CC_NVTX("cc_kl_target_argmax");
  CC_REQUIRE(target && out && target_rows >= 0 && num_cards > 0 && ldt >= num_cards, "cc_kl_target_argmax: bad arguments");
  if (target_rows == 0) return CC_OK;
  kl_target_argmax_kernel<<<target_rows, 256, 0, as_stream(stream)>>>(target, ldt, num_cards, out);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// row_hit (nullable, int32 [rows]) with target_argmax (int32, one entry per target row, cc_kl_target_argmax): 1 where
// the first maximal logit of the row is the target row's argmax -- Keras' categorical_accuracy on the softmax output
// (metrics=['accuracy'], src/ml/train.py:87).  Persistent kernels only (dbias != NULL).
int cc_softmax_kl_fwd_bwd_metrics(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                                  int32_t rows, int32_t num_cards, int32_t ncols_pad, double grad_scale, float* dz,
                                  int64_t lddz, double* row_loss, int round_tf32, float* dbias, void* dz_bf16,
                                  int64_t lddz_bf16, const double* tlogt, const int32_t* target_argmax, int32_t* row_hit,
                                  void* stream) {
  CC_NVTX("cc_softmax_kl_fwd_bwd_ex");
  CC_REQUIRE((row_hit == nullptr) || (target_argmax && dbias),
             "cc_softmax_kl_fwd_bwd: row_hit needs target_argmax and the persistent kernel (dbias != NULL)");
  CC_REQUIRE(!tlogt || dbias, "cc_softmax_kl_fwd_bwd: the target table is used by the persistent kernel only (dbias != NULL)");
  CC_REQUIRE(z && target && row_loss, "cc_softmax_kl_fwd_bwd: null pointer");
  CC_REQUIRE(!dz_bf16 || (dbias && lddz_bf16 >= ncols_pad && lddz_bf16 % 4 == 0 && (reinterpret_cast<uintptr_t>(dz_bf16) & 7) == 0),
             "cc_softmax_kl_fwd_bwd: bf16 dlogits need the persistent kernel (dbias != NULL), lddz_bf16 %% 4 == 0 >= ncols_pad");
  __nv_bfloat16* dz16 = static_cast<__nv_bfloat16*>(dz_bf16);
  if (dz16 && !dz) { dz = const_cast<float*>(z); lddz = ldz; }      // (unused: the kernel writes dz16 only)
  CC_REQUIRE(num_cards > 0 && ncols_pad >= num_cards, "cc_softmax_kl_fwd_bwd: bad sizes");
  CC_REQUIRE(!dz || lddz >= ncols_pad, "cc_softmax_kl_fwd_bwd: lddz too small");
  cudaStream_t st = as_stream(stream);
  if (dbias) {
    CC_REQUIRE(dz && cc_softmax_kl_fuses_dbias(num_cards, ncols_pad, ldz, ldt, lddz) &&
                   ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(target) | reinterpret_cast<uintptr_t>(dz)) % 16 == 0),
               "cc_softmax_kl_fwd_bwd: dbias needs the persistent kernel (see cc_softmax_kl_fuses_dbias) and 16-byte aligned buffers");
    CC_CHECK_CUDA(cudaMemsetAsync(dbias, 0, size_t(num_cards) * sizeof(float), st));
    if (rows == 0) return CC_OK;
    const size_t smem = size_t(num_cards) * 8;
    const int grid = rows < sm_count() ? rows : sm_count();
    auto fits = [&](int threads, int iters) { return (ncols_pad >> 2) <= (iters + 1) * threads && (num_cards >> 2) <= iters * threads; };
    const bool fits768 = fits(768, 7) && g_kl_variant != 2, fits512 = fits(512, 11);
    if ((fits768 || fits512) && g_kl_variant != 1) {
#define CC_KL_REGS(FAST_, RT_, THREADS_, ITERS_)                                                                      \
      do {                                                                                                            \
        CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_regs_kernel<FAST_, THREADS_, ITERS_>,                            \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                  \
        softmax_kl_regs_kernel<FAST_, THREADS_, ITERS_><<<grid, THREADS_, smem, st>>>(                                 \
            z, ldz, target, ldt, target_rows, rows, num_cards, ncols_pad, float(grad_scale), dz, lddz, row_loss, RT_,  \
            dbias, dz16, lddz_bf16, tlogt, target_argmax, row_hit);                                                   \
      } while (0)
      if (fits768) { if (round_tf32) CC_KL_REGS(true, dz16 ? 0 : 1, 768, 7); else CC_KL_REGS(false, 0, 768, 7); }
      else         { if (round_tf32) CC_KL_REGS(true, dz16 ? 0 : 1, 512, 11); else CC_KL_REGS(false, 0, 512, 11); }
#undef CC_KL_REGS
    } else if (round_tf32) {
      CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_persistent_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      softmax_kl_persistent_kernel<true><<<grid, KLP_THREADS, smem, st>>>(z, ldz, target, ldt, target_rows, rows, num_cards,
                                                                         ncols_pad, float(grad_scale), dz, lddz, row_loss,
                                                                         dz16 ? 0 : 1, dbias, dz16, lddz_bf16, tlogt, target_argmax, row_hit);
    } else {
      CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_persistent_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      softmax_kl_persistent_kernel<false><<<grid, KLP_THREADS, smem, st>>>(z, ldz, target, ldt, target_rows, rows, num_cards,
                                                                          ncols_pad, float(grad_scale), dz, lddz, row_loss, 0, dbias,
                                                                          dz16, lddz_bf16, tlogt, target_argmax, row_hit);
    }
    CC_CHECK_LAUNCH();
    return CC_OK;
  }
  if (rows == 0) return CC_OK;
  const size_t cache_bytes = size_t(num_cards) * 2 * sizeof(float);
  const bool aligned = (num_cards % 4 == 0) && (ldz % 4 == 0) && (ldt % 4 == 0) && (ncols_pad % 4 == 0) &&
                       (!dz || lddz % 4 == 0) &&
                       ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(target) | reinterpret_cast<uintptr_t>(dz)) % 16 == 0);
  if (aligned && size_t(num_cards) * 4 <= 100 * 1024) {
    const size_t smem = size_t(num_cards) * 4;
    if (round_tf32) {
      CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_rows_fast_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      softmax_kl_rows_fast_kernel<true><<<rows, KL_THREADS, smem, st>>>(z, ldz, target, ldt, target_rows, num_cards, ncols_pad,
                                                                       float(grad_scale), dz, lddz, row_loss, 1);
    } else {
      CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_rows_fast_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      softmax_kl_rows_fast_kernel<false><<<rows, KL_THREADS, smem, st>>>(z, ldz, target, ldt, target_rows, num_cards, ncols_pad,
                                                                        float(grad_scale), dz, lddz, row_loss, 0);
    }
  } else if (cache_bytes <= 200 * 1024) {
    CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)cache_bytes));
    softmax_kl_rows_kernel<true><<<rows, 1024, cache_bytes, st>>>(z, ldz, target, ldt, target_rows, num_cards,
                                                                 ncols_pad, float(grad_scale), dz, lddz, row_loss, round_tf32);
  } else {
    softmax_kl_rows_kernel<false><<<rows, 1024, 0, st>>>(z, ldz, target, ldt, target_rows, num_cards, ncols_pad,
                                                         float(grad_scale), dz, lddz, row_loss, round_tf32);
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// Loss-only softmax-KL for evaluation: row_loss (and, with target_argmax, row_hit) exactly as
// cc_softmax_kl_fwd_bwd_metrics computes them with the same tlogt and fast (= its round_tf32) flag; z is only read.
// Register-resident kernel shapes only (num_cards % 4 == 0, num_cards <= 22 528, 16-byte aligned rows).
int cc_softmax_kl_loss(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                       int32_t rows, int32_t num_cards, int32_t ncols_pad, const double* tlogt,
                       const int32_t* target_argmax, double* row_loss, int32_t* row_hit, int fast, void* stream) {
  CC_NVTX("cc_softmax_kl_loss");
  CC_REQUIRE(z && target && row_loss, "cc_softmax_kl_loss: null pointer");
  CC_REQUIRE(!target_argmax == !row_hit, "cc_softmax_kl_loss: target_argmax and row_hit are given together");
  CC_REQUIRE(rows >= 0 && num_cards > 0 && ncols_pad >= num_cards, "cc_softmax_kl_loss: bad sizes");
  auto fits = [&](int threads, int iters) { return (ncols_pad >> 2) <= (iters + 1) * threads && (num_cards >> 2) <= iters * threads; };
  const bool fits768 = fits(768, 7) && g_kl_variant != 2, fits512 = fits(512, 11);
  CC_REQUIRE(num_cards % 4 == 0 && ldz % 4 == 0 && ldt % 4 == 0 && ncols_pad % 4 == 0 && (fits768 || fits512) &&
                 ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(target)) % 16 == 0),
             "cc_softmax_kl_loss: num_cards %d outside the register kernel's shapes (num_cards %% 4 == 0, <= 22528, "
             "16-byte aligned rows)", num_cards);
  if (rows == 0) return CC_OK;
  cudaStream_t st = as_stream(stream);
  const size_t smem = size_t(num_cards) * 8;
  const int grid = rows < sm_count() ? rows : sm_count();
#define CC_KL_LOSS(FAST_, THREADS_, ITERS_)                                                                             \
  do {                                                                                                                \
    CC_CHECK_CUDA(cudaFuncSetAttribute(softmax_kl_regs_kernel<FAST_, THREADS_, ITERS_, false>,                        \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                      \
    softmax_kl_regs_kernel<FAST_, THREADS_, ITERS_, false><<<grid, THREADS_, smem, st>>>(                             \
        z, ldz, target, ldt, target_rows, rows, num_cards, ncols_pad, 0.f, nullptr, 0, row_loss, 0, nullptr, nullptr, \
        0, tlogt, target_argmax, row_hit);                                                                            \
  } while (0)
  if (fits768) { if (fast) CC_KL_LOSS(true, 768, 7); else CC_KL_LOSS(false, 768, 7); }
  else         { if (fast) CC_KL_LOSS(true, 512, 11); else CC_KL_LOSS(false, 512, 11); }
#undef CC_KL_LOSS
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_loss_finalize(const double* bce_rows, int32_t nb, double bce_div, const double* kl_rows, int32_t nr,
                     double kl_div, double reg, double* out3, void* stream) {
  CC_NVTX("cc_loss_finalize");
  CC_REQUIRE(out3 && (nb == 0 || bce_rows) && (nr == 0 || kl_rows), "cc_loss_finalize: null pointer");
  loss_finalize_kernel<<<1, 1024, 0, as_stream(stream)>>>(bce_rows, nb, bce_div, kl_rows, nr, kl_div, reg, out3);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_adam_step(float* params, const float* grads, float* m, float* v, int64_t n, const int64_t* step_ptr, float lr,
                 float beta1, float beta2, float eps, float* shadow_tf32, void* stream) {
  CC_NVTX("cc_adam_step");
  CC_REQUIRE(params && grads && m && v && step_ptr && n >= 0, "cc_adam_step: bad arguments");
  CC_REQUIRE((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(m) |
              reinterpret_cast<uintptr_t>(v)) % 16 == 0, "cc_adam_step: buffers must be 16-byte aligned");
  if (n == 0) return CC_OK;
  const int64_t threads = ceil_div<int64_t>(n, 4);
  adam_kernel<<<(unsigned)ceil_div<int64_t>(threads, 256), 256, 0, as_stream(stream)>>>(params, grads, m, v, n, step_ptr,
                                                                                      lr, beta1, beta2, eps, shadow_tf32);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_adam_step_p2p(const void* const* grads_ptrs, void* const* params_ptrs, int world, int rank, float* m, float* v,
                     int64_t lo, int64_t hi, const int64_t* step_ptr, float lr, float beta1, float beta2, float eps,
                     const void* grads_multicast, void* params_multicast, void* stream) {
  CC_NVTX("cc_adam_step_p2p");
  CC_REQUIRE(grads_ptrs && params_ptrs && m && v && step_ptr, "cc_adam_step_p2p: null pointer");
  CC_REQUIRE(world >= 1 && world <= P2P_MAX_WORLD && rank >= 0 && rank < world, "cc_adam_step_p2p: bad world/rank");
  CC_REQUIRE(lo >= 0 && hi >= lo && lo % 4 == 0 && hi % 4 == 0, "cc_adam_step_p2p: the slice must be 4-element aligned");
  CC_REQUIRE((grads_multicast == nullptr) == (params_multicast == nullptr),
             "cc_adam_step_p2p: give both multicast pointers or neither");
  PeerPtrs pp{};
  for (int r = 0; r < world; ++r) {
    CC_REQUIRE(grads_ptrs[r] && params_ptrs[r] &&
                   ((reinterpret_cast<uintptr_t>(grads_ptrs[r]) | reinterpret_cast<uintptr_t>(params_ptrs[r])) & 15) == 0,
               "cc_adam_step_p2p: rank %d buffers must be non-null and 16-byte aligned", r);
    pp.grads[r] = static_cast<const float*>(grads_ptrs[r]);
    pp.params[r] = static_cast<float*>(params_ptrs[r]);
  }
  pp.grads_mc = static_cast<const float*>(grads_multicast);
  pp.params_mc = static_cast<float*>(params_multicast);
  CC_REQUIRE(((reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(grads_multicast) |
               reinterpret_cast<uintptr_t>(params_multicast)) & 15) == 0,
             "cc_adam_step_p2p: m, v and the multicast pointers must be 16-byte aligned");
  if (hi == lo) return CC_OK;
  const int64_t threads = (hi - lo) / 4;
  cudaStream_t st = as_stream(stream);
  // float4 per thread: 4 on the multicast path, 2 for <= 4 ranks, 1 above (must match U in the kernel)
#define CC_P2P_LAUNCH(CAP, MC)                                                                                   \
  adam_p2p_kernel<CAP, MC><<<(unsigned)ceil_div<int64_t>(threads, 256 * ((MC) ? 4 : ((CAP) <= 4 ? 2 : 1))), 256, 0, st>>>( \
      pp, world, rank, m, v, lo, hi, step_ptr, lr, beta1, beta2, eps)
  if (grads_multicast) CC_P2P_LAUNCH(2, true);
  else if (world <= 2) CC_P2P_LAUNCH(2, false);
  else if (world <= 4) CC_P2P_LAUNCH(4, false);
  else if (world <= 8) CC_P2P_LAUNCH(8, false);
  else CC_P2P_LAUNCH(16, false);
#undef CC_P2P_LAUNCH
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_convert_f32_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int32_t rows, int32_t cols, void* stream) {
  CC_NVTX("cc_convert_f32_bf16");
  CC_REQUIRE(src && dst && rows >= 0 && cols >= 0 && ld_src >= cols && ld_dst >= cols, "cc_convert_f32_bf16: bad arguments");
  CC_REQUIRE(cols % 4 == 0 && ld_src % 4 == 0 && ld_dst % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(dst) & 7) == 0,
             "cc_convert_f32_bf16: cols and leading dimensions must be multiples of 4, buffers 16/8-byte aligned");
  if (rows == 0 || cols == 0) return CC_OK;
  const int64_t total = int64_t(rows) * (cols / 4);
  convert_f32_bf16_kernel<<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, as_stream(stream)>>>(
      src, ld_src, static_cast<__nv_bfloat16*>(dst), ld_dst, rows, cols / 4);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_round_tf32(const float* x, float* out, int64_t n, void* stream) {
  CC_NVTX("cc_round_tf32");
  CC_REQUIRE(x && out && n >= 0, "cc_round_tf32: bad arguments");
  if (n == 0) return CC_OK;
  round_tf32_kernel<<<(unsigned)ceil_div<int64_t>(n, 256), 256, 0, as_stream(stream)>>>(x, out, n);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

int cc_sigmoid_f32(const float* z, float* out, int64_t n, void* stream) {
  CC_NVTX("cc_sigmoid_f32");
  CC_REQUIRE(z && out && n >= 0, "cc_sigmoid_f32: bad arguments");
  if (n == 0) return CC_OK;
  sigmoid_kernel<<<(unsigned)ceil_div<int64_t>(n, 256), 256, 0, as_stream(stream)>>>(z, out, n);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

}  // extern "C"
