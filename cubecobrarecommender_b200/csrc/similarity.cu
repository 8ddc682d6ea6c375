// Card and cube similarity for many queries at once: the -cosine distance of every (query, candidate) pair of 64-d
// encoder embeddings, bit for bit the value cosine_neg_kernel (topn.cu) writes for that pair, so the batched table,
// `similar()` and the single-card CLI agree on every near tie.  The rows are ranked afterwards by the masked select
// (cc_topn_masked_f32, ascending).
//
// cosine_neg_kernel gives lane l (0..31) of a warp the partial p_l = fmaf(a[l+32], b[l+32], fmaf(a[l], b[l], 0)) and
// sums the 32 partials with warp_sum's xor butterfly (offsets 16, 8, 4, 2, 1), which hands every lane the same tree:
// node(L, S) = node(L, 2S) + node(L + S, 2S) with leaves node(l, 32) = p_l and the sum node(0, 1).  One thread evaluates
// that tree depth-first here (sim_tree), with at most five pending partials per pair, for a 4 x 4 register tile of
// pairs; the inverse norms rsqrtf(fmaxf(x.x, 1e-12)) come from the same tree once per row, and the distance is
// -((ab * rsqrt_q) * rsqrt_c) as in cosine_neg_kernel.  Every add and multiply is an explicit _rn intrinsic, so nvcc
// cannot contract a product into a sum and change a bit.
#include "cc_common.cuh"

namespace cc {

constexpr int SIM_DIM = 64;                 // the encoder's bottleneck width; the only dim the tree is written for
constexpr int SIM_TILE = 64;                // queries and candidates per CTA
constexpr int SIM_T = 4;                    // per thread: SIM_T queries x SIM_T candidates
constexpr int SIM_THREADS = (SIM_TILE / SIM_T) * (SIM_TILE / SIM_T);

// node(L, S) of warp_sum's butterfly for N independent sums at once; leaf(l, p) writes the N partials p_l
template <int L, int S, int N, class Leaf>
__device__ __forceinline__ void sim_tree(const Leaf& leaf, float (&v)[N]) {
  if constexpr (S == 32) {
    leaf(L, v);
  } else {
    float w[N];
    sim_tree<L, 2 * S>(leaf, v);
    sim_tree<L + S, 2 * S>(leaf, w);
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __fadd_rn(v[i], w[i]);
  }
}

// CTA (x, y): candidates [64 x, 64 x + 64) against queries [64 y, ...) (y strides by gridDim.y).  Rows are staged
// k-major in shared memory (qs[k][row]), so a thread's four queries (or candidates) at one k are one float4; rows past
// the end are zero and never written out.
__global__ void __launch_bounds__(SIM_THREADS, 2)
cosine_neg_many_kernel(const float* __restrict__ queries, int64_t ldq, int32_t num_queries,
                       const float* __restrict__ cands, int64_t ldc, int32_t num_cands, float* __restrict__ out,
                       int64_t ldo, int vec_out) {
  __shared__ __align__(16) float qs[SIM_DIM][SIM_TILE];
  __shared__ __align__(16) float cs[SIM_DIM][SIM_TILE];
  __shared__ __align__(16) float qn[SIM_TILE];
  __shared__ __align__(16) float cn[SIM_TILE];
  const int tid = threadIdx.x;
  const int tx = tid % (SIM_TILE / SIM_T), ty = tid / (SIM_TILE / SIM_T);
  const int c0 = blockIdx.x * SIM_TILE;
  const int q_tiles = (num_queries + SIM_TILE - 1) / SIM_TILE;
  for (int qt = blockIdx.y; qt < q_tiles; qt += gridDim.y) {
    const int q0 = qt * SIM_TILE;
    // stage: thread t loads float4 column f of row t % 64 (consecutive lanes -> consecutive rows: conflict-free
    // transposed stores)
    {
      const int r = tid % SIM_TILE;
#pragma unroll
      for (int f = tid / SIM_TILE; f < SIM_DIM / 4; f += SIM_THREADS / SIM_TILE) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        if (q0 + r < num_queries) a = *reinterpret_cast<const float4*>(queries + int64_t(q0 + r) * ldq + 4 * f);
        if (c0 + r < num_cands) b = *reinterpret_cast<const float4*>(cands + int64_t(c0 + r) * ldc + 4 * f);
        qs[4 * f][r] = a.x; qs[4 * f + 1][r] = a.y; qs[4 * f + 2][r] = a.z; qs[4 * f + 3][r] = a.w;
        cs[4 * f][r] = b.x; cs[4 * f + 1][r] = b.y; cs[4 * f + 2][r] = b.z; cs[4 * f + 3][r] = b.w;
      }
    }
    __syncthreads();
    if (tid < 2 * SIM_TILE) {                 // one row's inverse norm per thread: the same tree over x * x
      const float(*xs)[SIM_TILE] = tid < SIM_TILE ? qs : cs;
      const int r = tid % SIM_TILE;
      float s[1];
      sim_tree<0, 1>([&](int l, float(&p)[1]) {
        const float x0 = xs[l][r], x1 = xs[l + 32][r];
        p[0] = fmaf(x1, x1, fmaf(x0, x0, 0.f));
      }, s);
      (tid < SIM_TILE ? qn : cn)[r] = rsqrtf(fmaxf(s[0], 1e-12f));
    }
    float ab[SIM_T * SIM_T];
    sim_tree<0, 1>([&](int l, float(&p)[SIM_T * SIM_T]) {
      const float4 a0 = *reinterpret_cast<const float4*>(&qs[l][SIM_T * ty]);
      const float4 a1 = *reinterpret_cast<const float4*>(&qs[l + 32][SIM_T * ty]);
      const float4 b0 = *reinterpret_cast<const float4*>(&cs[l][SIM_T * tx]);
      const float4 b1 = *reinterpret_cast<const float4*>(&cs[l + 32][SIM_T * tx]);
      const float x0[SIM_T] = {a0.x, a0.y, a0.z, a0.w}, x1[SIM_T] = {a1.x, a1.y, a1.z, a1.w};
      const float y0[SIM_T] = {b0.x, b0.y, b0.z, b0.w}, y1[SIM_T] = {b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < SIM_T; ++i)
#pragma unroll
        for (int j = 0; j < SIM_T; ++j) p[i * SIM_T + j] = fmaf(x1[i], y1[j], fmaf(x0[i], y0[j], 0.f));
    }, ab);
    __syncthreads();                          // norms written; every thread is done reading qs / cs
    const float4 cnv = *reinterpret_cast<const float4*>(&cn[SIM_T * tx]);
    const float cinv[SIM_T] = {cnv.x, cnv.y, cnv.z, cnv.w};
    const int c = c0 + SIM_T * tx;
#pragma unroll
    for (int i = 0; i < SIM_T; ++i) {
      const int q = q0 + SIM_T * ty + i;
      if (q >= num_queries) break;
      const float qinv = qn[SIM_T * ty + i];
      float d[SIM_T];
#pragma unroll
      for (int j = 0; j < SIM_T; ++j) d[j] = -__fmul_rn(__fmul_rn(ab[i * SIM_T + j], qinv), cinv[j]);
      float* o = out + int64_t(q) * ldo + c;
      if (vec_out && c + SIM_T <= num_cands) {
        *reinterpret_cast<float4*>(o) = make_float4(d[0], d[1], d[2], d[3]);
      } else {
#pragma unroll
        for (int j = 0; j < SIM_T; ++j)
          if (c + j < num_cands) o[j] = d[j];
      }
    }
    __syncthreads();                          // qn / cn and the tiles are rewritten by the next query tile
  }
}

}  // namespace cc

using namespace cc;

extern "C" {

int cc_cosine_neg_many_f32(const float* queries, int64_t ldq, int32_t num_queries, const float* cands, int64_t ldc,
                           int32_t num_cands, int32_t dim, float* out, int64_t ldo, void* stream) {
  CC_NVTX("cc_cosine_neg_many_f32");
  CC_REQUIRE(queries && cands && out, "cc_cosine_neg_many_f32: null pointer");
  CC_REQUIRE(dim == SIM_DIM, "cc_cosine_neg_many_f32: dim must be %d (the encoder's width), got %d", SIM_DIM, dim);
  CC_REQUIRE(num_queries >= 0 && num_cands > 0 && ldq >= dim && ldc >= dim && ldo >= num_cands,
             "cc_cosine_neg_many_f32: bad sizes");
  CC_REQUIRE((ldq & 3) == 0 && (ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(queries) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(cands) & 15) == 0,
             "cc_cosine_neg_many_f32: queries and cands need 16-byte aligned rows (16-byte aligned bases, ldq and ldc "
             "multiples of 4)");
  if (num_queries == 0) return CC_OK;
  const int q_tiles = ceil_div(num_queries, SIM_TILE);
  const dim3 grid(ceil_div(num_cands, SIM_TILE), q_tiles < 65535 ? q_tiles : 65535);
  const int vec_out = (ldo & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  cosine_neg_many_kernel<<<grid, SIM_THREADS, 0, as_stream(stream)>>>(queries, ldq, num_queries, cands, ldc,
                                                                      num_cands, out, ldo, vec_out);
  CC_CHECK_LAUNCH();
  return CC_OK;
}

}  // extern "C"
