// tcgen05 tensor-core GEMM for sm_100a: TMA-fed, TMEM accumulators, fused epilogues.
//
// Replaces the dense matmuls behind the Dense layers of reference src/ml/model.py:27-33,
// 58-64 and their gradients, and carries the sigmoid-BCE loss of src/ml/train.py:85-86
// inside the epilogue of the 512 -> C decoder GEMM, so the C-wide logits never reach HBM
// (only dlogits do).
//
//   C[M,N] = epi(op(A) op(B)),   fp32 storage, kind::tf32 (10-bit mantissa products, fp32
//   accumulation in TMEM) or bf16 storage, kind::f16.
//
// Structure (one persistent CTA per SM, 256 threads):
//   warp 0   TMA producer: cp.async.bulk.tensor boxes -> 128B-swizzled smem ring
//   warp 1   MMA issuer : one elected lane issues tcgen05.mma (128 x BN x 8|16), commits to
//            the stage's "empty" mbarrier and, per tile, to the accumulator's "full" barrier
//   warp 2   TMEM allocator (2 accumulator buffers: MMA of tile i+1 overlaps epilogue of tile i)
//   warps 4-11 epilogue: tcgen05.ld 32 lanes x 32 columns -> bias/ReLU/mask or BCE -> swizzled
//            smem staging -> TMA store (or TMA reduce-add for split-K), so global writes are
//            full 128-byte lines issued by the copy engine, not by the warps
// Operands may be K-major ([rows, K], K contiguous) or MN-major ([K, rows], rows contiguous);
// both are loaded with 128B-swizzle boxes and described to the MMA by shared-memory matrix
// descriptors (LBO/SBO as in the PTX ISA "canonical layouts").
// Tile = 128 x BN with BN in {128, 256}: with 4-byte operands a 128x128 tile needs 32 KB of
// L2->SM traffic per MFLOP and saturates L2 bandwidth near 380 TFLOP/s; 128x256 cuts that by 25%.
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>

#include "cc_common.cuh"

namespace cc {
namespace tc {

constexpr int BM = 128;
constexpr int NUM_ACC = 2;
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 128 + 32 * EPI_WARPS;           // warps 0-3: TMA producer, MMA issuer, TMEM allocator, idle
constexpr int STAGE_A_BYTES = BM * 128;                 // 128 rows x one 128-byte swizzle row
constexpr int EPI_STAGE_BYTES = EPI_WARPS * 4096;       // one (32 rows x 128 B) staging buffer per epilogue warp
constexpr int BAR_BYTES = 256;

// CTAS = 2: a CTA pair (cluster of two SMs of one TPC) works on a 256 x BN tile with
// tcgen05.mma.cta_group::2 -- each CTA stages its own 128 rows of A and only HALF of the B tile
// (BN/2 rows), so the L2->SM operand traffic per flop drops by a third at BN = 256.
template <int BN, int CTAS> struct Cfg {
  static constexpr int STAGE_B_BYTES = (BN / CTAS) * 128;
  static constexpr int STAGE_BYTES = STAGE_A_BYTES + STAGE_B_BYTES;
  static constexpr int STAGES = STAGE_BYTES >= 49152 ? 4 : 6;
  static constexpr int TMEM_COLS = NUM_ACC * BN;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_STAGE_BYTES + BAR_BYTES + 1024 /*align slack*/;
};

// EPI_BCE16: the fused sigmoid-BCE epilogue writing dlogits as bf16 (they feed the bf16 dW / dX GEMMs of the "bf16" mode)
// EPI_BCE_ACC / EPI_BCE16_ACC: the same two with the Keras binary_accuracy count (four more instructions per element,
// compiled in only when the caller asks for metrics)
// EPI_BCE_LOSS / EPI_BCE_LOSS_ACC: loss (and accuracy) partials only, for evaluation: no dlogits, no C tensor map, no
// bias-gradient sums
enum Epilogue : int { EPI_STORE = 0, EPI_BCE = 1, EPI_COUNT = 2, EPI_BCE16 = 3, EPI_BCE_ACC = 4, EPI_BCE16_ACC = 5,
                      EPI_BCE_LOSS = 6, EPI_BCE_LOSS_ACC = 7 };
// operand kinds: fp32 storage / kind::tf32, bf16 storage / kind::f16, uint8 storage / kind::i8 (int32 accumulators:
// the co-occurrence contraction X^T X over 0/1 bytes is exact)
enum Kind : int { KIND_TF32 = 0, KIND_BF16 = 1, KIND_U8 = 2 };

struct Params {
  int m, n, k;
  int m_tiles, n_tiles, k_blocks;       // k_blocks per split
  int split_k, total_k_blocks;
  const float* bias;
  const float* mask; long long ldmask;
  int relu, reduce_add, round_tf32;
  int n_store;                           // columns the store map covers (EPI_BCE: ldc, pad columns get zeros)
  // EPI_BCE
  const uint32_t* ybits; long long ywords;
  float inv_count;
  double* loss_partial;                  // [tiles][EPI_WARPS]
  double* acc_partial;                   // nullable, same layout: number of cells with round(sigmoid(z)) == y (Keras binary_accuracy)
  float* dbias;                          // EPI_BCE: column sums of dlogits (= the output layer's bias gradient), atomically added
  int a_mn_major, b_mn_major;
  int a_mn3, b_mn3;                      // the MN-major operand is described by a 3-D tensor map (make_map_mn3): one TMA per k-block
  int* sched;                            // {next-tile counter, finished units}: self-resetting (see TileRing)
  // hybrid stream-K (static scheduling only): the first dp_tiles output tiles are walked round-robin with their whole
  // K range and stored; the LAST sk_tiles tiles are cut along K into num_units contiguous spans of k-blocks, one per
  // unit, and every span is TMA-reduce-added into the (pre-zeroed) tile.  sk_tiles = 0: off.
  int dp_tiles, sk_tiles;
  // tile order of the plain GEMM: 0 = tile row fastest (tile = mt + m_tiles * nt), 1 = tile column fastest.  The tiles
  // that run at the same time should share operand panels: with many tile rows and only 2-4 tile columns (dW1 =
  // x^T g1: 82 x 2) row-fastest order puts the two tiles that read the SAME 4.2 MB panel of x a whole wave apart, and
  // the panel comes from DRAM twice (ncu: 702 MB read for 353 MB of operands); column-fastest makes them neighbours.
  int nt_fastest;
  // EPI_COUNT: C = A A^T is symmetric -> only tiles with nt >= mt are computed (square 256 x 256 pair tiles) and every
  // off-diagonal tile is also written transposed
  int symmetric;
  int* count_out; long long ldcount;
  // tile order of the symmetric GEMM: bands of `band_rows` tile rows; inside a band column by column, all the band's
  // rows of a column before the next column.  The band's A row blocks (band_rows x 256 cards x K bytes) stay in L2
  // and every B column block is fetched from DRAM once per BAND instead of once per ROW (ncu: 13.3 GB -> see DESIGN)
  int band_rows;
  int band_start[72];                    // first tile index of each band (host-computed), band_start[n_bands] = total
};

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  uint32_t spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    if (done) break;
    if (++spins > (1u << 28)) __trap();      // watchdog: a protocol bug must not hang the GPU
  }
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// ---- CTA-pair (cluster of 2) helpers
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load issued by either CTA of a pair; completion bytes are credited to a barrier that may live in the
// peer CTA (the leader's "full" barrier), hence the cluster-space barrier address and .cta_group::2
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}

// 3-D forms (see make_map_mn3): one instruction fetches every 32-float column group of an MN-major tf32 operand
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {   // acquire at cluster scope
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    if (done) break;
    if (++spins > (1u << 28)) __trap();
  }
}
__device__ __forceinline__ void st_shared_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}

// ---- dynamic tile scheduler ------------------------------------------------------------------------------
// Tiles are handed out at run time: unit u (a CTA, or a CTA pair) starts on tile u and then draws further tiles
// from a global atomic counter, so a unit that starts late or shares its SM (an NCCL all_reduce overlapping
// backward) simply takes fewer tiles instead of stretching the whole kernel.  One scheduler thread per unit
// (warp 3 of the leader CTA) publishes tile ids through a small shared-memory ring to the unit's TMA producer(s),
// MMA issuer and epilogue warps; -1 ends the kernel.  The counters reset themselves: the unit that draws the last
// terminal value zeroes them for the next launch.
constexpr int SCHED_DEPTH = 4;
struct TileRing {
  uint64_t* full;        // [SCHED_DEPTH]  scheduler -> consumers (count 1)
  uint64_t* empty;       // [SCHED_DEPTH]  consumers -> scheduler (lives in the leader CTA)
  volatile int* ids;     // [SCHED_DEPTH]
  uint32_t empty_cluster_addr;   // leader's `empty` array in cluster address space (pairs), 0 otherwise
  int slot; uint32_t phase;
};
template <int CTAS>
__device__ __forceinline__ int ring_next(TileRing& r) {
  if (CTAS == 2) mbar_wait_cluster(&r.full[r.slot], r.phase); else mbar_wait(&r.full[r.slot], r.phase);
  const int t = r.ids[r.slot];
  if (CTAS == 2) mbar_arrive_cluster(r.empty_cluster_addr + r.slot * 8); else mbar_arrive(&r.empty[r.slot]);
  if (++r.slot == SCHED_DEPTH) { r.slot = 0; r.phase ^= 1; }
  return t;
}

template <int CTAS>
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
  if (CTAS == 2) {   // arrives on the barrier at this offset in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
  } else {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
  }
}
#define CC_TCGEN05_MMA(GROUP, KINDSTR)                                                                  \
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"                                      \
               "tcgen05.mma.cta_group::" GROUP ".kind::" KINDSTR " [%0], %1, %2, %3, p;\n\t}"            \
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory")
template <int KIND, int CTAS>
__device__ __forceinline__ void tcgen05_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  if (CTAS == 2) {
    if (KIND == KIND_BF16) CC_TCGEN05_MMA("2", "f16");
    else if (KIND == KIND_U8) CC_TCGEN05_MMA("2", "i8");
    else CC_TCGEN05_MMA("2", "tf32");
  } else {
    if (KIND == KIND_BF16) CC_TCGEN05_MMA("1", "f16");
    else if (KIND == KIND_U8) CC_TCGEN05_MMA("1", "i8");
    else CC_TCGEN05_MMA("1", "tf32");
  }
}
#undef CC_TCGEN05_MMA
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ float exp2f_approx(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float lg2_approx(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// shared-memory matrix descriptor (version 1)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                             uint32_t layout_type) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr >> 4) & 0x3fffu);
  d |= uint64_t((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= uint64_t(1) << 46;             // descriptor version (Blackwell)
  d |= uint64_t(layout_type) << 61;   // 2 = SWIZZLE_128B (16-byte atoms), 1 = SWIZZLE_128B with 32-byte atoms
  return d;
}

// ------------------------------------------------------------------------ kernel
// upper-triangle tiles (nt >= mt) of the symmetric count GEMM in banded order (see Params::band_rows)
__device__ __forceinline__ void decode_tile(const Params& p, int tile, int& mt, int& nt, int& ks) {
  if (p.symmetric) {
    const int n = p.n_tiles, g = p.band_rows;
    int b = 0;
    while (p.band_start[b + 1] <= tile) ++b;               // <= 71 bands
    const int r0 = b * g;
    const int rows = min(g, n - r0);                        // tile rows in this band
    int t = tile - p.band_start[b];
    const int tri = rows * (rows + 1) / 2;                  // the band's first `rows` columns form a triangle
    if (t < tri) {
      int j = 0;
      while ((j + 1) * (j + 2) / 2 <= t) ++j;               // column j of the triangle holds rows 0..j
      mt = r0 + (t - j * (j + 1) / 2); nt = r0 + j;
    } else {
      t -= tri;
      nt = r0 + rows + t / rows; mt = r0 + t % rows;
    }
    ks = 0;
  } else {
    if (p.nt_fastest) {
      nt = tile % p.n_tiles;
      mt = (tile / p.n_tiles) % p.m_tiles;
    } else {
      mt = tile % p.m_tiles;
      nt = (tile / p.m_tiles) % p.n_tiles;
    }
    ks = tile / (p.m_tiles * p.n_tiles);
  }
}

// One unit's walk over its work in hybrid stream-K mode: its share of the data-parallel tiles first, then its span of
// the stream-K tiles' k-blocks (which may cover the tail of one tile, whole tiles, and the head of another).  Every
// role of the CTA (TMA producer, MMA issuer, epilogue warps) runs the same walk.
struct SkWalk {
  int dp_next; long long cur, hi;
  __device__ __forceinline__ void init(const Params& p, int unit, int num_units) {
    dp_next = unit;
    const long long total = (long long)p.sk_tiles * p.total_k_blocks;
    cur = total * unit / num_units;
    hi = total * (unit + 1) / num_units;
  }
  __device__ __forceinline__ bool next(const Params& p, int num_units, int& tile, int& kb0, int& kb1) {
    if (dp_next < p.dp_tiles) { tile = dp_next; dp_next += num_units; kb0 = 0; kb1 = p.total_k_blocks; return true; }
    if (cur < hi) {
      const int t = int(cur / p.total_k_blocks);
      kb0 = int(cur - (long long)t * p.total_k_blocks);
      const long long left = hi - cur;
      kb1 = (long long)(p.total_k_blocks - kb0) <= left ? p.total_k_blocks : kb0 + int(left);
      tile = p.dp_tiles + t;
      cur += kb1 - kb0;
      return true;
    }
    return false;
  }
};

template <int KIND, int EPI, int BN, int CTAS>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const __grid_constant__ CUtensorMap map_c, const Params p) {
  using C = Cfg<BN, CTAS>;
  constexpr bool BF16 = KIND == KIND_BF16;
  constexpr bool LOSS_ONLY = EPI == EPI_BCE_LOSS || EPI == EPI_BCE_LOSS_ACC;      // nothing is stored but the partials
  constexpr bool IS_BCE = EPI == EPI_BCE || EPI == EPI_BCE16 || EPI == EPI_BCE_ACC || EPI == EPI_BCE16_ACC || LOSS_ONLY;
  constexpr bool OUT16 = EPI == EPI_BCE16 || EPI == EPI_BCE16_ACC;   // output elements are bf16 (32 x 32 block = 64-byte rows)
  constexpr bool WANT_ACC = EPI == EPI_BCE_ACC || EPI == EPI_BCE16_ACC || EPI == EPI_BCE_LOSS_ACC;
  constexpr int BN_LOAD = BN / CTAS;             // rows of the B tile this CTA stages
  constexpr int STAGES = C::STAGES;
  constexpr int STAGE_BYTES = C::STAGE_BYTES;
  constexpr int ELEM = KIND == KIND_U8 ? 1 : (BF16 ? 2 : 4);
  constexpr int BK = 128 / ELEM;                 // elements per 128-byte swizzle row (32 | 64 | 128)
  constexpr int UMMA_K = 32 / ELEM;              // 8 | 16 | 32
  constexpr int MMAS_PER_STAGE = BK / UMMA_K;    // 4
  constexpr int MN_BOX = BK;                     // MN-major boxes are [BK rows(k)] x [BK elems (128 B)]
  constexpr int MN_BOX_BYTES = BK * 128;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* epi_smem = smem + STAGES * STAGE_BYTES;                       // 1024-byte aligned
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_smem + EPI_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + NUM_ACC;
  uint64_t* sched_full = tmem_empty + NUM_ACC;
  uint64_t* sched_empty = sched_full + SCHED_DEPTH;
  int* sched_ids = reinterpret_cast<int*>(sched_empty + SCHED_DEPTH);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sched_ids + SCHED_DEPTH);

  // Programmatic dependent launch: let the NEXT kernel of the stream be scheduled as soon as every CTA of this grid
  // is running; its CTAs take whatever SMs are (or become) free, run their prologue (barrier init, TMEM
  // allocation, descriptor prefetch) and park at griddepcontrol.wait below until this grid has completed.  The step
  // is a chain of ~35 GEMM launches, most of them a few microseconds long: this hides launch latency and prologue.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tiles of (BM*CTAS) x BN; the symmetric count GEMM only visits the upper triangle of its square tile grid
  const int total_tiles = p.symmetric ? (p.n_tiles * (p.n_tiles + 1)) / 2 : p.m_tiles * p.n_tiles * p.split_k;
  const int cta_rank = CTAS == 2 ? int(cluster_ctarank()) : 0;
  const int unit = CTAS == 2 ? int(blockIdx.x >> 1) : int(blockIdx.x);       // scheduling unit: CTA or CTA pair
  const int num_units = CTAS == 2 ? int(gridDim.x >> 1) : int(gridDim.x);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    if constexpr (!LOSS_ONLY) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < NUM_ACC; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], EPI_WARPS * CTAS); }
    // ring consumers: per CTA its TMA producer and epilogue warps, plus the leader's MMA issuer
    for (int d = 0; d < SCHED_DEPTH; ++d) { mbar_init(&sched_full[d], 1); mbar_init(&sched_empty[d], (1 + EPI_WARPS) * CTAS + 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (CTAS == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(C::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(C::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tcgen05_fence_before();
  if (CTAS == 2) cluster_sync_all();      // the peer's barriers are initialised before anything signals them
  else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // nothing above touched global memory; everything below may read what the previous kernel wrote (activations,
  // parameters, scheduler counters) or overwrite what it still reads
  asm volatile("griddepcontrol.wait;" ::: "memory");
  TileRing ring{sched_full, sched_empty, sched_ids, CTAS == 2 ? mapa_shared(smem_u32(sched_empty), 0) : 0u, 0, 0u};
  const bool dynamic = p.sched != nullptr;
  // static mode: unit u walks tiles u, u + num_units, ... with no ring traffic at all
  auto next_tile = [&](int cur) -> int {
    if (dynamic) return ring_next<CTAS>(ring);
    const int t = cur < 0 ? unit : cur + num_units;
    return t < total_tiles ? t : -1;
  };
  const bool stream_k = p.sk_tiles > 0;         // (never together with the dynamic scheduler or the symmetric GEMM)
  SkWalk walk;
  walk.init(p, unit, num_units);
  // next piece of work for the calling role: tile (-1: done) and its k-block range
  auto next_work = [&](int& tile, int& kb0, int& kb1) {
    if (stream_k) {
      if (!walk.next(p, num_units, tile, kb0, kb1)) tile = -1;
      return;
    }
    tile = next_tile(tile);
    if (tile < 0) return;
    int mt_, nt_, ks_;
    decode_tile(p, tile, mt_, nt_, ks_);
    kb0 = ks_ * p.k_blocks;
    kb1 = min(kb0 + p.k_blocks, p.total_k_blocks);
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int tile = -1, kb0 = 0, kb1 = 0;
      for (next_work(tile, kb0, kb1); tile >= 0; next_work(tile, kb0, kb1)) {
        int mt, nt, ks;
        decode_tile(p, tile, mt, nt, ks);
        const int a_row0 = (mt * CTAS + cta_rank) * BM;             // this CTA's 128 rows of the (pair) tile
        const int b_row0 = nt * BN + cta_rank * BN_LOAD;            // and its share of the B tile
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          uint8_t* sb = sa + STAGE_A_BYTES;
          if (CTAS == 2) {
            // both CTAs' boxes are credited to the LEADER's full barrier (the MMA issuer waits there)
            const uint32_t bar = mapa_shared(smem_u32(&full_bar[stage]), 0);
            if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2 * STAGE_BYTES);
            if (p.a_mn3) {
              tma_load_3d_pair(sa, &map_a, bar, 0, kb * BK, a_row0 / MN_BOX);
            } else if (p.a_mn_major) {
#pragma unroll
              for (int j = 0; j < BM / MN_BOX; ++j)
                tma_load_2d_pair(sa + j * MN_BOX_BYTES, &map_a, bar, a_row0 + j * MN_BOX, kb * BK);
            } else {
              tma_load_2d_pair(sa, &map_a, bar, kb * BK, a_row0);
            }
            if (p.b_mn3) {
              tma_load_3d_pair(sb, &map_b, bar, 0, kb * BK, b_row0 / MN_BOX);
            } else if (p.b_mn_major) {
#pragma unroll
              for (int j = 0; j < BN_LOAD / MN_BOX; ++j)
                tma_load_2d_pair(sb + j * MN_BOX_BYTES, &map_b, bar, b_row0 + j * MN_BOX, kb * BK);
            } else {
              tma_load_2d_pair(sb, &map_b, bar, kb * BK, b_row0);
            }
          } else {
            mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
            if (p.a_mn3) {
              tma_load_3d(sa, &map_a, &full_bar[stage], 0, kb * BK, a_row0 / MN_BOX);
            } else if (p.a_mn_major) {
#pragma unroll
              for (int j = 0; j < BM / MN_BOX; ++j)
                tma_load_2d(sa + j * MN_BOX_BYTES, &map_a, &full_bar[stage], a_row0 + j * MN_BOX, kb * BK);
            } else {
              tma_load_2d(sa, &map_a, &full_bar[stage], kb * BK, a_row0);
            }
            if (p.b_mn3) {
              tma_load_3d(sb, &map_b, &full_bar[stage], 0, kb * BK, b_row0 / MN_BOX);
            } else if (p.b_mn_major) {
#pragma unroll
              for (int j = 0; j < BN / MN_BOX; ++j)
                tma_load_2d(sb + j * MN_BOX_BYTES, &map_b, &full_bar[stage], b_row0 + j * MN_BOX, kb * BK);
            } else {
              tma_load_2d(sb, &map_b, &full_bar[stage], kb * BK, b_row0);
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && cta_rank == 0) {       // in a pair only the leader CTA issues (cta_group::2 drives both SMs)
      // instruction descriptor: D format (1 = f32, 2 = s32), A/B formats (tf32 = 2, bf16 = 1, u8 = 0), major-ness, N, M
      constexpr uint32_t FMT = KIND == KIND_TF32 ? 2u : (KIND == KIND_BF16 ? 1u : 0u);
      const uint32_t idesc = ((KIND == KIND_U8 ? 2u : 1u) << 4) | (FMT << 7) | (FMT << 10) |
                             (uint32_t(p.a_mn_major) << 15) | (uint32_t(p.b_mn_major) << 16) |
                             (uint32_t(BN >> 3) << 17) | (uint32_t((BM * CTAS) >> 4) << 24);
      // K-major: rows 128 B apart, 8-row groups 1024 B apart (SBO); K advance 32 B inside the swizzle row.
      // MN-major: 128-byte MN atoms LBO apart, k-row groups SBO apart; K advance UMMA_K rows.
      // 32-bit (tf32) MN-major operands only exist in the "128B swizzle, 32-byte atom" layout: atoms of 4 k-rows
      // (SBO = 512 B); every other case uses the plain 128B swizzle with 8-row atoms (SBO = 1024 B).
      const uint32_t a_lbo = p.a_mn_major ? MN_BOX_BYTES : 16, b_lbo = p.b_mn_major ? MN_BOX_BYTES : 16;
      const uint32_t a_lt = (KIND == KIND_TF32 && p.a_mn_major) ? 1u : 2u, b_lt = (KIND == KIND_TF32 && p.b_mn_major) ? 1u : 2u;
      const uint32_t a_sbo = a_lt == 1u ? 512u : 1024u, b_sbo = b_lt == 1u ? 512u : 1024u;
      const uint32_t a_kstep = p.a_mn_major ? UMMA_K * 128 : 32, b_kstep = p.b_mn_major ? UMMA_K * 128 : 32;
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      int tile = -1, kb0 = 0, kb1 = 0;
      for (next_work(tile, kb0, kb1); tile >= 0; next_work(tile, kb0, kb1)) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + STAGE_A_BYTES;
#pragma unroll
          for (int k = 0; k < MMAS_PER_STAGE; ++k) {
            const uint64_t adesc = make_desc(sa + k * a_kstep, a_lbo, a_sbo, a_lt);
            const uint64_t bdesc = make_desc(sb + k * b_kstep, b_lbo, b_sbo, b_lt);
            tcgen05_mma<KIND, CTAS>(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          tcgen05_commit<CTAS>(&empty_bar[stage]);    // frees the smem slot (in both CTAs) when these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        tcgen05_commit<CTAS>(&tmem_full[acc]);        // accumulator complete -> epilogue (of both CTAs)
        if (++acc == NUM_ACC) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp == 3) {
    // ===================== tile scheduler (leader CTA only) =====================
    if (lane == 0 && cta_rank == 0 && dynamic) {
      const uint32_t peer_ids = CTAS == 2 ? mapa_shared(smem_u32(sched_ids), 1) : 0u;
      const uint32_t peer_full = CTAS == 2 ? mapa_shared(smem_u32(sched_full), 1) : 0u;
      int slot = 0; uint32_t phase = 0;
      int tile = unit < total_tiles ? unit : -1;
      while (true) {
        if (CTAS == 2) mbar_wait_cluster(&sched_empty[slot], phase ^ 1); else mbar_wait(&sched_empty[slot], phase ^ 1);
        sched_ids[slot] = tile;
        if (CTAS == 2) {
          st_shared_cluster_u32(peer_ids + slot * 4, uint32_t(tile));
          mbar_arrive_cluster(peer_full + slot * 8);           // release.cluster: orders the store above
        }
        mbar_arrive(&sched_full[slot]);
        if (tile < 0) break;
        if (++slot == SCHED_DEPTH) { slot = 0; phase ^= 1; }
        tile = num_units + atomicAdd(p.sched, 1);
        if (tile >= total_tiles) {
          tile = -1;
          // every unit draws exactly one terminal value; the last one to do so re-arms the counters
          if (atomicAdd(p.sched + 1, 1) == num_units - 1) { p.sched[0] = 0; p.sched[1] = 0; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps) =====================
    // A warp may only read the TMEM lane quarter warp % 4, so warps w and w + 4 share a 32-row quarter and split
    // the tile's columns in halves.  Two epilogue warps per scheduler hide each other's latencies (TMEM loads,
    // MUFU chains, staging-buffer turnaround); with one warp per scheduler the fused BCE epilogue was the
    // bottleneck of its GEMM (16 us per 128 x 256 tile against 10 us for the MMAs).
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;
    constexpr int NCH = BN / 64;                            // 32-column chunks per warp
    uint8_t* sbuf = epi_smem + (warp - 4) * 4096;           // one 4 KB staging buffer (32 rows x 128 B, 128B-swizzled)
    int acc = 0; uint32_t acc_phase = 0;
    const uint32_t leader_tmem_empty = CTAS == 2 ? mapa_shared(smem_u32(&tmem_empty[0]), 0) : 0u;
    int tile = -1, wkb0 = 0, wkb1 = 0;
    while (true) {
      if (dynamic) {
        if (lane == 0) tile = ring_next<CTAS>(ring);
        tile = __shfl_sync(0xffffffffu, tile, 0);
      } else {
        next_work(tile, wkb0, wkb1);
      }
      if (tile < 0) break;
      int mt, nt, ks;
      decode_tile(p, tile, mt, nt, ks);
      const bool has_k = stream_k ? (wkb0 < wkb1) : (ks * p.k_blocks < p.total_k_blocks);
      // a stream-K span that does not cover its tile's whole K range is one of several contributions to it
      const bool red_add = p.reduce_add || (stream_k && (wkb0 != 0 || wkb1 != p.total_k_blocks));
      const int row0 = (mt * CTAS + cta_rank) * BM + q * 32;
      const int row = row0 + lane;
      const bool row_ok = row < p.m;
      const int colw = nt * BN + half * (BN / 2);           // first column of this warp's half of the tile
      // operands of the epilogue that live in global memory (the bias slice, and for BCE this row's y bits: NCH
      // consecutive words) are fetched for the warp's whole half tile while its MMAs still run, so no chunk waits
      // on a global load.  Lane l holds the bias of column col0 + l; element j gets it by shuffle from lane j.
      float bias_r[NCH];
      uint32_t y_r[NCH];
#pragma unroll
      for (int cb = 0; cb < NCH; ++cb) {
        const int col = colw + cb * 32 + lane;
        bias_r[cb] = (p.bias && col < p.n) ? __ldg(p.bias + col) : 0.f;
        y_r[cb] = 0u;
      }
      if (IS_BCE && row_ok) {
        const uint32_t* yrow = p.ybits + (long long)row * p.ywords + (colw >> 5);
        const bool in_range = colw + BN / 2 <= p.ywords * 32;
        if (NCH == 4 && in_range && ((reinterpret_cast<uintptr_t>(yrow) & 15) == 0)) {
          const uint4 w = __ldg(reinterpret_cast<const uint4*>(yrow));
          y_r[0] = w.x; y_r[1] = w.y; y_r[NCH > 2 ? 2 : 0] = w.z; y_r[NCH > 2 ? 3 : 0] = w.w;
        } else {
#pragma unroll
          for (int cb = 0; cb < NCH; ++cb)
            if (colw + cb * 32 < p.n_store) y_r[cb] = __ldg(yrow + cb);
        }
      }
      const float inv_row = row_ok ? p.inv_count : 0.f;     // rows beyond m: zero gradient (they feed the column sums)
      mbar_wait(&tmem_full[acc], acc_phase);
      tcgen05_fence_after();
      float row_loss = 0.f, row_hits = 0.f;
      // The BCE body is long (a rolled loop keeps it inside the instruction cache: unrolling it 8x cost 300 -> 442 us),
      // so the prefetched registers are ROTATED instead of indexed; the short store body is fully unrolled.
#pragma unroll(IS_BCE ? 1 : NCH)
      for (int cb = 0; cb < NCH; ++cb) {
        const int col0 = colw + cb * 32;
        if (col0 >= p.n_store || row0 >= p.m || !has_k) break;      // warp-uniform
        uint32_t v[32];
        __syncwarp();
        tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * BN + half * (BN / 2) + cb * 32), v);
        const float b_cur = bias_r[0];
        const uint32_t ybw = y_r[0];
#pragma unroll
        for (int r = 0; r + 1 < NCH; ++r) { bias_r[r] = bias_r[r + 1]; y_r[r] = y_r[r + 1]; }
        float out[32];
        if (EPI == EPI_COUNT) {
          // int32 accumulators pass through bit for bit; an off-diagonal tile is also written transposed
          // (for a fixed column the 32 lanes hold 32 consecutive rows -> one 128-byte line per store)
#pragma unroll
          for (int j = 0; j < 32; ++j) out[j] = __uint_as_float(v[j]);
          if (p.symmetric && nt != mt && row_ok) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (col0 + j < p.n) {
                int* dst = p.count_out + (long long)(col0 + j) * p.ldcount + row;
                if (p.reduce_add) atomicAdd(dst, int(v[j]));
                else *dst = int(v[j]);
              }
            }
          }
        } else if (IS_BCE) {
          // softplus(z) - z*y and sigmoid(z) from one exp: e = exp(-|z|) (ex2, rcp: 2 MUFU ops per element).  The
          // log terms of a chunk are taken together: sum_j log(1 + e_j) = log(prod_j (1 + e_j)) -- every factor lies in
          // (1, 2], so the product of 32 stays below 2^32 and costs one multiply per element and ONE lg2 per chunk
          // instead of a lg2 and a multiply-add per element (relative error of the product <= 32 ulps: 2e-6 in a sum of
          // order 10)
          float prod = 1.f;
          auto bce_elem = [&](int j, bool live, float& g) {
            const float z = __uint_as_float(v[j]) + __shfl_sync(0xffffffffu, b_cur, j);
            const float y = float((ybw >> j) & 1u);
            if constexpr (WANT_ACC) {                        // round(sigmoid(z)) == y: sigmoid(0) = 0.5 rounds to 0 (half to even)
              const float hit = ((z > 0.f) == (y != 0.f)) ? 1.f : 0.f;
              row_hits += live ? hit : 0.f;
            }
            const float e = exp2f_approx(-1.4426950408889634f * fabsf(z));
            const float s1 = 1.f + e;
            const float r = LOSS_ONLY ? 0.f : rcp_approx(s1);
            const float lin = fmaf(-z, y, fmaxf(z, 0.f));
            row_loss += live ? lin : 0.f;
            prod *= live ? s1 : 1.f;
            if constexpr (!LOSS_ONLY) g = ((z >= 0.f ? r : e * r) - y) * inv_row;
          };
          if (col0 + 32 <= p.n) {                       // warp-uniform: only the last column tile is ragged
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float g;
              bce_elem(j, true, g);
              if constexpr (!LOSS_ONLY) out[j] = p.round_tf32 ? rn_tf32_bits(g) : g;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float g;
              const bool live = (col0 + j < p.n);
              bce_elem(j, live, g);
              if constexpr (!LOSS_ONLY) {
                g = live ? g : 0.f;
                out[j] = p.round_tf32 ? rn_tf32_bits(g) : g;
              }
            }
          }
          row_loss = fmaf(0.6931471805599453f, lg2_approx(prod), row_loss);
          if constexpr (LOSS_ONLY) continue;
        } else {
          // branch-free inner loops: bias is 0 when absent, ReLU is a max with -inf when off
          const float floor_v = p.relu ? 0.f : -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            out[j] = fmaxf(__uint_as_float(v[j]) + __shfl_sync(0xffffffffu, b_cur, j), floor_v);
          if (p.mask) {           // ReLU backward: keep the gradient where the forward activation was positive
            if (row_ok) {
              const float* mrow = p.mask + (long long)row * p.ldmask + col0;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < p.n) out[j] = (__ldg(mrow + j) > 0.f) ? out[j] : 0.f;
            }
          }
          if (p.round_tf32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) out[j] = rn_tf32_bits(out[j]);
          }
        }
        // registers -> swizzled staging (row = lane, 16-byte chunk c at position c ^ (lane & 7)) -> TMA store
        if (lane == 0) tma_wait_group_read<0>();        // the store that last read this buffer has drained
        __syncwarp();
        if (OUT16) {
          // bf16 block: plain row-major 64-byte rows (the C tensor map is unswizzled with a 32 x 32 box)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const __nv_bfloat162 h = __floats2bfloat162_rn(out[8 * c + 2 * e], out[8 * c + 2 * e + 1]);
              w[e] = *reinterpret_cast<const uint32_t*>(&h);
            }
            *reinterpret_cast<uint4*>(sbuf + lane * 64 + (c << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        } else {
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<float4*>(sbuf + lane * 128 + ((c ^ (lane & 7)) << 4)) =
                make_float4(out[4 * c], out[4 * c + 1], out[4 * c + 2], out[4 * c + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (red_add) tma_reduce_add_2d(&map_c, sbuf, col0, row0);
          else              tma_store_2d(&map_c, sbuf, col0, row0);
          tma_commit_group();
        }
        if (IS_BCE && p.dbias) {
          // bias gradient = column sums of dlogits: lane j adds up column j of the staged 32 x 32 block (for a fixed
          // row the 32 lanes hit 32 different banks of the swizzled row -- or, bf16, 16 banks two lanes a word) and
          // issues one coalesced RED per chunk.  Rows beyond m and columns beyond n hold zeros.
          float cs = 0.f;
#pragma unroll
          for (int r = 0; r < 32; ++r) {
            if (OUT16) cs += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(sbuf + r * 64 + (lane << 1)));
            else cs += *reinterpret_cast<const float*>(sbuf + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + ((lane & 3) << 2));
          }
          if (col0 + lane < p.n) atomicAdd(p.dbias + col0 + lane, cs);
        }
      }
      if (IS_BCE) {
        // one float64 partial per (tile, warp): fixed summation order downstream
        const float s = row_ok ? row_loss : 0.f;
        const double d = warp_sum(double(s));
        if (lane == 0) p.loss_partial[((long long)tile * CTAS + cta_rank) * EPI_WARPS + (warp - 4)] = d;
        if (WANT_ACC && p.acc_partial) {                  // warp-uniform
          const double a = warp_sum(double(row_ok ? row_hits : 0.f));
          if (lane == 0) p.acc_partial[((long long)tile * CTAS + cta_rank) * EPI_WARPS + (warp - 4)] = a;
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CTAS == 2) mbar_arrive_cluster(leader_tmem_empty + acc * 8);   // the leader's issuer waits for both CTAs
        else mbar_arrive(&tmem_empty[acc]);
      }
      if (++acc == NUM_ACC) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all stores complete before exit
  }

  tcgen05_fence_before();
  if (CTAS == 2) cluster_sync_all();      // neither CTA may retire while the other can still signal its barriers
  else __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    if (CTAS == 2)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::TMEM_COLS) : "memory");
  }
}

// elementwise epilogue for split-K GEMMs whose epilogue is not linear: c = round(mask(relu(c + bias)))
__global__ void post_epilogue_kernel(float* __restrict__ c, long long ldc, int m, int n, const float* __restrict__ bias,
                                     int relu, const float* __restrict__ mask, long long ldmask, int round_tf32) {
  // lets a dependent tcgen05 GEMM / chain launch (programmatic stream serialisation) be scheduled and run its prologue
  // while this grid drains; it still waits (griddepcontrol.wait) for this grid's completion before touching memory
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)m * n) return;
  const int r = int(i / n), col = int(i % n);
  float z = c[(long long)r * ldc + col];
  if (bias) z += bias[col];
  if (relu) z = fmaxf(z, 0.f);
  if (mask) z = (mask[(long long)r * ldmask + col] > 0.f) ? z : 0.f;
  if (round_tf32) z = rn_tf32(z);
  c[(long long)r * ldc + col] = z;
}

// ---------------------------------------------------------------- host helpers
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

// 2-D row-major matrix [rows][cols] (cols contiguous, leading dimension ld elements);
// box = box_rows x (128 bytes of columns), 128B swizzle (32-byte atoms for 4-byte MN-major operands).
enum MapType : int { MAP_F32 = 0, MAP_BF16 = 1, MAP_U8 = 2, MAP_S32 = 3 };
static int make_map(CUtensorMap* map, const void* base, int elem, int mtype, long long rows, long long cols,
                    long long ld, int box_rows, bool atom32, int box_cols = 0 /* 0: 128 bytes, swizzled; else unswizzled */) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return CC_ERR_CUDA; }
  cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  cuuint64_t strides[1] = {cuuint64_t(ld) * elem};
  cuuint32_t box[2] = {cuuint32_t(box_cols ? box_cols : 128 / elem), cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = mtype == MAP_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : mtype == MAP_U8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                 : mtype == MAP_S32 ? CU_TENSOR_MAP_DATA_TYPE_INT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const CUresult r = fn(map, dt, 2,
                        const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        box_cols ? CU_TENSOR_MAP_SWIZZLE_NONE
                                 : (atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B),
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): base=%p rows=%lld cols=%lld ld=%lld", int(r), base, rows, cols, ld);
    return CC_ERR_CUDA;
  }
  return CC_OK;
}

// An MN-major tf32 operand ([K][MN] row-major, MN contiguous) lands in shared memory as consecutive 4 KB boxes of
// [32 k-rows] x [32 floats] (128B swizzle with 32-byte atoms), one per 32-float column group.  As 2-D boxes that is 4-8
// TMA instructions per operand per k-block -- measured 5-18% slower than the same GEMM on K-major operands (one box),
// profiles/r02/gemm_layout_bench.jsonl: the producer's issue rate, not the MMA.  Described as a 3-D tensor
// {32 floats, K rows (stride ld), MN/32 groups (stride 128 bytes)} with a box of {32, 32, groups}, ONE instruction writes
// the same bytes to the same places.  The last group of a row may extend past MN (MN % 32 != 0): it then reads the
// first floats of the next row, which only ever feed output rows / columns that the store clips -- the caller makes
// sure those bytes exist (ld >= MN rounded up to 32, or the matrix is followed by more of the same buffer).
static int make_map_mn3(CUtensorMap* map, const void* base, long long k_rows, long long mn, long long ld, int groups) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return CC_ERR_CUDA; }
  cuuint64_t dims[3] = {32, cuuint64_t(k_rows), cuuint64_t((mn + 31) / 32)};
  cuuint64_t strides[2] = {cuuint64_t(ld) * 4, 128};
  cuuint32_t box[3] = {32, 32, cuuint32_t(groups)};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (3-D MN-major) failed (%d): base=%p k=%lld mn=%lld ld=%lld", int(r), base, k_rows, mn, ld);
    return CC_ERR_CUDA;
  }
  return CC_OK;
}

struct Problem {
  int transa, transb, m, n, k;
  const void* a; long long lda;
  const void* b; long long ldb;
  float* c; long long ldc;
  int kind;
};

// waves-based efficiency of (BN, split, CTA pairing) on `sms` SMs: with ctas = 2 the scheduling
// unit is a 256 x bn tile on one of sms/2 CTA pairs
static double plan_eff(int m, int n, int kblocks, int bn, int split, int sms, int ctas) {
  const int units = sms / ctas;
  const long long tiles = (long long)ceil_div(m, BM * ctas) * ceil_div(n, bn) * split;
  const int kb = ceil_div(kblocks, split);
  const long long waves = ceil_div<long long>(tiles, (long long)units);
  // a tile costs kb*bn (+ a fixed prologue/epilogue worth ~6 k-blocks); rows beyond m are wasted work
  const double busy = double(m) / (BM * ctas) * ceil_div(n, bn) * kblocks * bn;
  const double span = double(waves) * units * (kb + 6) * bn;
  double eff = busy / span;
  // L2->SM operand bytes per flop: 128x128 tiles are bandwidth-limited with 4-byte operands, 128x256 less so,
  // a 256x256 pair tile moves a third less than that
  if (ctas == 1) eff *= (bn == 128 ? 0.68 : 0.80);
  if (split > 1) eff *= 0.97;       // reduce traffic + zero fill
  return eff;
}

// Scheduler counters: a per-device pool of {next tile, finished units} pairs, handed out round-robin so GEMMs that
// are in flight at the same time (other streams) never share a pair; each pair zeroes itself when its launch ends.
constexpr int SCHED_POOL = 4096;
static int* sched_slot() {
  static int* pools[64] = {nullptr};
  static std::atomic<unsigned> next[64];
  static std::mutex mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  {
    std::lock_guard<std::mutex> lk(mu);
    if (!pools[dev]) {
      int* ptr = nullptr;
      if (cudaMalloc(&ptr, SCHED_POOL * 2 * sizeof(int)) != cudaSuccess) return nullptr;
      if (cudaMemset(ptr, 0, SCHED_POOL * 2 * sizeof(int)) != cudaSuccess) return nullptr;
      pools[dev] = ptr;
    }
  }
  return pools[dev] + 2 * (next[dev].fetch_add(1) % SCHED_POOL);
}

// Hybrid stream-K plan: how many of the m_tiles x n_tiles output tiles (the last ones) are cut along K and spread over
// all `units`.  Whole waves of tiles stay data-parallel (stored once, no reduction); what does not fill a wave -- the
// 16 left-over tiles of the 164-tile dW pass on 74 CTA pairs, or all 32 tiles of the long-K dX pass -- is spread evenly,
// so no unit idles through a ragged last wave and only those tiles pay read-modify-write traffic (with plain split-K
// EVERY tile is reduce-added split_k times: ncu showed 131 MB written for a 42.8 MB dW).  0 = plain data-parallel.
// Only for long-K passes (>= 64 k-blocks): a short-K pass loses little to its ragged wave and its spans would be all
// prologue.
static int stream_k_tiles(int m_tiles, int n_tiles, int k_blocks, int units) {
  const int t = m_tiles * n_tiles;
  if (units <= 0 || k_blocks < 64) return 0;
  const int full = t / units, rem = t - full * units;
  if (rem == 0) return 0;
  int sk = rem;
  // spans shorter than ~16 k-blocks are all prologue/epilogue: fold one full wave into the stream-K part instead
  if (full >= 1 && (long long)rem * k_blocks / units < 16) sk = rem + units;
  if (sk > t) sk = t;
  // not worth it when the stream-K part is nearly a full wave anyway (the ragged wave wastes < 10%)
  if (full >= 1 && rem * 10 >= units * 9) return 0;
  return sk;
}

// programmatic dependent launch of consecutive GEMMs (cc_gemm_tc_set_pdl; on by default, CC_GEMM_PDL=0 disables)
static int g_pdl = getenv("CC_GEMM_PDL") ? atoi(getenv("CC_GEMM_PDL")) : 1;

// 0 = static round-robin tiles (default: on an undisturbed GPU it is ~3% faster, nothing is claimed ahead),
// 1 = dynamic tile scheduler (cc_gemm_tc_set_dynamic_tiles; the data-parallel engine turns it on while all_reduces
// overlap backward and steal SMs)
static int g_dynamic_tiles = 0;

// -1 = planner decides, 0 = never pair, 1 = always pair (cc_gemm_tc_set_pair_mode; experiments and tests)
static int g_pair_mode = -1;

// -1 = planner decides between plain split-K and hybrid stream-K, 0 = never stream-K, 1 = stream-K whenever the tile count
// leaves a ragged wave (cc_gemm_tc_set_stream_k; tests and A/B measurements)
static int g_stream_k = getenv("CC_GEMM_STREAM_K") ? atoi(getenv("CC_GEMM_STREAM_K")) : -1;

// -1 = column-fastest tile order where it saves operand re-reads (see Params::nt_fastest), 0 = always row-fastest
// (CC_GEMM_TILE_ORDER=0; A/B measurements)
static int g_tile_order = getenv("CC_GEMM_TILE_ORDER") ? atoi(getenv("CC_GEMM_TILE_ORDER")) : -1;

// 1 = MN-major tf32 operands through 3-D tensor maps (one TMA per operand per k-block, see make_map_mn3), 0 = 2-D boxes
// (CC_GEMM_MN3=0; A/B measurements)
static int g_mn3 = getenv("CC_GEMM_MN3") ? atoi(getenv("CC_GEMM_MN3")) : 1;
static std::atomic<long long> g_mn3_used{0};       // operands described by 3-D maps so far (cc_gemm_tc_mn3_count)
// memory ranges the caller has declared fully readable (cc_gemm_tc_register_readable): an MN-major operand whose rows
// are not padded to 32 floats may still take the 3-D form when the bytes behind its ragged last column group lie
// inside such a range (a Keras kernel inside the flat parameter buffer is followed by its bias)
static std::mutex g_readable_mu;
static uintptr_t g_readable[32][2];
static int g_readable_n = 0;
static int g_use_readable = getenv("CC_GEMM_READABLE") ? atoi(getenv("CC_GEMM_READABLE")) : 1;   // 0: ignore the registered ranges (A/B)
static bool readable_range(const void* base, long long k_rows, long long mn, long long ld) {
  if (!g_use_readable) return false;
  const uintptr_t lo = reinterpret_cast<uintptr_t>(base);
  const uintptr_t hi = lo + (uintptr_t(k_rows - 1) * uintptr_t(ld) + uintptr_t((mn + 31) / 32 * 32)) * 4;
  std::lock_guard<std::mutex> lk(g_readable_mu);
  for (int i = 0; i < g_readable_n; ++i)
    if (lo >= g_readable[i][0] && hi <= g_readable[i][1]) return true;
  return false;
}

// the waves model of plan_eff for the hybrid stream-K schedule of (bn, ctas): full data-parallel waves, then every
// unit's span of the stream-K k-blocks (two partial tiles' worth of prologue/epilogue)
static double plan_eff_sk(int m, int n, int kblocks, int bn, int sms, int ctas) {
  const int units = sms / ctas;
  const int mt = ceil_div(m, BM * ctas), nt = ceil_div(n, bn);
  const int sk = stream_k_tiles(mt, nt, kblocks, units);
  if (sk == 0) return -1.0;
  const int dp = mt * nt - sk;
  const long long span = (long long)ceil_div(dp, units) * (kblocks + 6) + ceil_div<long long>((long long)sk * kblocks, units) + 12;
  const double busy = double(m) / (BM * ctas) * nt * kblocks;
  double eff = busy / (double(units) * double(span));
  if (ctas == 1) eff *= (bn == 128 ? 0.68 : 0.80);
  return eff * 0.99;          // zero fill + reduce traffic of the stream-K tiles only
}

static int max_pair_clusters(const void* kern, int smem_bytes) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(unsigned(sm_count() / 2 * 2));
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = size_t(smem_bytes);
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

template <int KIND, int EPI, int BN, int CTAS>
static int launch_bn(const Problem& pr, Params p, cudaStream_t st) {
  using C = Cfg<BN, CTAS>;
  constexpr bool BF16 = KIND == KIND_BF16;
  constexpr bool TF32 = KIND == KIND_TF32;
  const int elem = KIND == KIND_U8 ? 1 : (BF16 ? 2 : 4);
  const int mt = KIND == KIND_U8 ? MAP_U8 : (BF16 ? MAP_BF16 : MAP_F32);
  const int bk = 128 / elem;
  CUtensorMap map_a, map_b, map_c;
  int rc;
  // transa=0: A is [M][K] (K-major)  -> box 128 rows x 128 B;  transa=1: A is [K][M] (MN-major) -> box bk rows x 128 B
  // (3-D MN-major maps: tf32 only, and only when the bytes behind a ragged last column group exist inside the row)
  p.a_mn3 = (TF32 && pr.transa && g_mn3 && (pr.m % 32 == 0 || pr.lda >= ((pr.m + 31) / 32) * 32 ||
                                            readable_range(pr.a, pr.k, pr.m, pr.lda))) ? 1 : 0;
  p.b_mn3 = (TF32 && !pr.transb && g_mn3 && (pr.n % 32 == 0 || pr.ldb >= ((pr.n + 31) / 32) * 32 ||
                                             readable_range(pr.b, pr.k, pr.n, pr.ldb))) ? 1 : 0;
  if (p.a_mn3 && make_map_mn3(&map_a, pr.a, pr.k, pr.m, pr.lda, BM / 32) != CC_OK) p.a_mn3 = 0;    // (driver refused: 2-D boxes)
  if (p.a_mn3)        { rc = CC_OK; ++g_mn3_used; }
  else if (pr.transa) rc = make_map(&map_a, pr.a, elem, mt, pr.k, pr.m, pr.lda, bk, TF32);
  else                rc = make_map(&map_a, pr.a, elem, mt, pr.m, pr.k, pr.lda, BM, false);
  if (rc != CC_OK) return rc;
  // transb=1: B is [N][K] (K-major);  transb=0: B is [K][N] (MN-major); a CTA of a pair loads BN/2 rows
  if (p.b_mn3 && make_map_mn3(&map_b, pr.b, pr.k, pr.n, pr.ldb, (BN / CTAS) / 32) != CC_OK) p.b_mn3 = 0;
  if (p.b_mn3)        { rc = CC_OK; ++g_mn3_used; }
  else if (pr.transb) rc = make_map(&map_b, pr.b, elem, mt, pr.n, pr.k, pr.ldb, BN / CTAS, false);
  else                rc = make_map(&map_b, pr.b, elem, mt, pr.k, pr.n, pr.ldb, bk, TF32);
  if (rc != CC_OK) return rc;
  // C: fp32 (int32 counts) [M][n_store] boxes of 32 rows x 32 columns (TMA clips rows >= M and columns >= n_store)
  if constexpr (EPI == EPI_BCE_LOSS || EPI == EPI_BCE_LOSS_ACC) { memset(&map_c, 0, sizeof(map_c)); rc = CC_OK; }   // never read
  else if (EPI == EPI_BCE16 || EPI == EPI_BCE16_ACC) rc = make_map(&map_c, pr.c, 2, MAP_BF16, pr.m, p.n_store, pr.ldc, 32, false, 32);
  else rc = make_map(&map_c, pr.c, 4, EPI == EPI_COUNT ? MAP_S32 : MAP_F32, pr.m, p.n_store, pr.ldc, 32, false);
  if (rc != CC_OK) return rc;
  p.a_mn_major = pr.transa ? 1 : 0;
  p.b_mn_major = pr.transb ? 0 : 1;
  p.m_tiles = ceil_div(pr.m, BM * CTAS);
  p.n_tiles = ceil_div(p.n_store, BN);
  p.total_k_blocks = ceil_div(pr.k, bk);
  if (p.split_k < 1) p.split_k = 1;
  p.k_blocks = ceil_div(p.total_k_blocks, p.split_k);
  p.split_k = ceil_div(p.total_k_blocks, p.k_blocks);
  int tiles = p.symmetric ? p.n_tiles * (p.n_tiles + 1) / 2 : p.m_tiles * p.n_tiles * p.split_k;
  p.sched = nullptr;
  if (g_dynamic_tiles) {
    p.sched = sched_slot();
    if (!p.sched) { set_error("cc_gemm_tc: could not allocate the tile-scheduler counters"); return CC_ERR_CUDA; }
  }
  auto kern = gemm_tc_kernel<KIND, EPI, BN, CTAS>;
  // per-device one-time setup (a process may drive several GPUs: one host thread or process per device)
  static std::mutex setup_mu;
  static bool attr_done[64] = {false};
  static int max_clusters_dev[64] = {0};
  int dev = 0;
  CC_CHECK_CUDA(cudaGetDevice(&dev));
  CC_REQUIRE(dev >= 0 && dev < 64, "cc_gemm_tc: device ordinal %d out of range", dev);
  {
    std::lock_guard<std::mutex> lk(setup_mu);
    if (!attr_done[dev]) {
      CC_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
      if (CTAS == 2) {
        int mc = max_pair_clusters(reinterpret_cast<const void*>(kern), C::SMEM_BYTES);
        if (mc <= 0) { set_error("cc_gemm_tc: no CTA-pair cluster can be resident (occupancy query)"); return CC_ERR_CUDA; }
        if (mc > sm_count() / 2) mc = sm_count() / 2;
        max_clusters_dev[dev] = mc;
      }
      attr_done[dev] = true;
    }
  }
  const int max_units = CTAS == 2 ? max_clusters_dev[dev] : sm_count();
  // hybrid stream-K (p.sk_tiles < 0 on entry = "choose"): see Params.  Only with static scheduling.
  if (p.sk_tiles < 0) {
    p.sk_tiles = 0;
    if (!p.symmetric && !p.sched && p.split_k == 1) p.sk_tiles = stream_k_tiles(p.m_tiles, p.n_tiles, p.total_k_blocks, max_units);
  }
  // column-fastest tile order (see Params): few tile columns, many tile rows, at least one full data-parallel wave
  p.nt_fastest = (!p.symmetric && g_tile_order != 0 && p.split_k == 1 && p.n_tiles < p.m_tiles && p.n_tiles <= 4 &&
                  p.m_tiles * p.n_tiles - (p.sk_tiles > 0 ? p.sk_tiles : 0) >= max_units) ? 1 : 0;
  p.dp_tiles = 0;
  if (p.sk_tiles > 0) {
    p.dp_tiles = p.m_tiles * p.n_tiles - p.sk_tiles;
    if (!p.reduce_add && p.nt_fastest) {
      // the stream-K tiles are the last sk_tiles of the column-fastest order: the right part of tile row mt0 (from tile
      // column nt0 on) and every row after it
      const int mt0 = p.dp_tiles / p.n_tiles, nt0 = p.dp_tiles % p.n_tiles;
      const long long row0 = (long long)mt0 * BM * CTAS, col0 = (long long)nt0 * BN;
      long long rowf = row0;                                 // first FULL stream-K row
      if (nt0 > 0 && row0 < pr.m) {
        const long long h = (row0 + BM * CTAS < pr.m ? BM * CTAS : pr.m - row0);
        if (col0 < p.n_store)
          CC_CHECK_CUDA(cudaMemset2DAsync(pr.c + row0 * pr.ldc + col0, size_t(pr.ldc) * 4, 0, size_t(p.n_store - col0) * 4, size_t(h), st));
        rowf = row0 + BM * CTAS;
      }
      if (rowf < pr.m)
        CC_CHECK_CUDA(cudaMemset2DAsync(pr.c + rowf * pr.ldc, size_t(pr.ldc) * 4, 0, size_t(p.n_store) * 4, size_t(pr.m - rowf), st));
    } else if (!p.reduce_add) {
      // the stream-K tiles are the last sk_tiles of the row-fastest tile order: the lower part of tile column nt0 (from
      // tile row mt0 on) and every column after it.  They are zeroed (two 2-D memsets); every span is reduce-added.
      const int nt0 = p.dp_tiles / p.m_tiles, mt0 = p.dp_tiles % p.m_tiles;
      const long long col0 = (long long)nt0 * BN, row0 = (long long)mt0 * BM * CTAS;
      long long colf = col0;                                 // first FULL stream-K column
      if (mt0 > 0 && col0 < p.n_store) {
        const long long w = (col0 + BN < p.n_store ? BN : p.n_store - col0);
        if (row0 < pr.m)
          CC_CHECK_CUDA(cudaMemset2DAsync(pr.c + row0 * pr.ldc + col0, size_t(pr.ldc) * 4, 0, size_t(w) * 4, size_t(pr.m - row0), st));
        colf = col0 + BN;
      }
      if (colf < p.n_store)
        CC_CHECK_CUDA(cudaMemset2DAsync(pr.c + colf, size_t(pr.ldc) * 4, 0, size_t(p.n_store - colf) * 4, pr.m, st));
    }
  }
  {
    int units = tiles < max_units ? tiles : max_units;
    if (p.sk_tiles > 0) {       // every unit takes a span of the stream-K k-blocks
      const long long iters = (long long)p.sk_tiles * p.total_k_blocks;
      units = iters < max_units ? int(iters) : max_units;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(CTAS * units));
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (g_pdl) {       // may start while the previous kernel of the stream drains (see griddepcontrol in the kernel)
      at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[na].val.programmaticStreamSerializationAllowed = 1;
      ++na;
    }
    if (CTAS == 2) {
      at[na].id = cudaLaunchAttributeClusterDimension;
      at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
      ++na;
    }
    cfg.attrs = at; cfg.numAttrs = na;
    CC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, map_a, map_b, map_c, p));
  }
  CC_CHECK_LAUNCH();
  return CC_OK;
}

template <int KIND, int EPI>
static int launch(const Problem& pr, Params p, int bn, int ctas, cudaStream_t st) {
  const int elem = KIND == KIND_U8 ? 1 : (KIND == KIND_BF16 ? 2 : 4);
  CC_REQUIRE((reinterpret_cast<uintptr_t>(pr.a) & 15) == 0 && (reinterpret_cast<uintptr_t>(pr.b) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(pr.c) & 15) == 0,
             "cc_gemm_tc: base pointers must be 16-byte aligned");
  CC_REQUIRE((pr.lda * elem) % 16 == 0 && (pr.ldb * elem) % 16 == 0 && (pr.ldc * ((EPI == EPI_BCE16 || EPI == EPI_BCE16_ACC) ? 2 : 4)) % 16 == 0,
             "cc_gemm_tc: leading dimensions must be multiples of 16 bytes (lda=%lld ldb=%lld ldc=%lld)", pr.lda,
             pr.ldb, pr.ldc);
  if (ctas == 2) return launch_bn<KIND, EPI, 256, 2>(pr, p, st);
  if (EPI == EPI_COUNT) { set_error("count GEMM runs on CTA pairs only"); return CC_ERR_ARGUMENT; }
  if (bn == 256) return launch_bn<KIND, EPI == EPI_COUNT ? EPI_STORE : EPI, 256, 1>(pr, p, st);
  return launch_bn<KIND, EPI == EPI_COUNT ? EPI_STORE : EPI, 128, 1>(pr, p, st);
}

// ------------------------------------------------------------------ co-occurrence counts on the tensor cores
// Bytes X^T[c][k - k0] = 1 for every card c of cube k of the chunk [k0, k0 + chunk): one warp per cube.
__global__ void expand_cubes_u8_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                       long long k0, int chunk, int num_cards, uint8_t* __restrict__ xt, long long ldx,
                                       int32_t* __restrict__ bad) {
  const int warps_per_block = blockDim.x >> 5;
  const int w = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  if (w >= chunk) return;
  const int lane = threadIdx.x & 31;
  const long long lo = indptr[k0 + w], hi = indptr[k0 + w + 1];
  for (long long i = lo + lane; i < hi; i += 32) {
    const int c = indices[i];
    if (c < 0 || c >= num_cards) { if (bad) atomicOr(bad, 1); continue; }
    xt[(long long)c * ldx + w] = 1;
  }
}


// ------------------------------------------------------------------ chain of small Dense layers in ONE kernel
// The 512 -> 256 -> 128 -> 64 (-> 128 -> 256 -> 512) layers around the 64-wide bottleneck are latency-bound as separate
// GEMMs (9-23 us each for a few hundred MFLOP; 27 of them are 18% of the step).  Here a CTA takes 128 rows through up to
// three consecutive layers without leaving the SM: layer 1 is an ordinary SS tcgen05.mma (A and B staged by TMA), its
// accumulator is turned into the next layer's operand IN TENSOR MEMORY (tcgen05.ld -> bias / ReLU or ReLU mask -> tf32
// rounding -> tcgen05.st to the same columns), and layers 2 and 3 are TS tcgen05.mma (A from tensor memory, B = the
// layer's kernel streamed through the same smem ring -- the producer runs ahead across layers).  Every layer's output
// is also written to global memory (swizzled staging -> TMA store): backward and the weight-gradient GEMMs need it.
// Same k order and the same fp32 accumulation as the separate GEMMs, so the results are bit-identical to them.
// Reference: the Dense stacks of src/ml/model.py:27-33, 58-64 (forward) and their input gradients (backward).
struct ChainLayer {
  int n, k;                 // output width (multiple of 64, <= 512) and reduction length (multiple of 32, <= 512)
  int b_mn_major;           // B = the layer's kernel: [K][N] row-major (forward, 1) or [N][K] row-major (backward, 0)
  int b_mn3;                // the MN-major kernel is described by a 3-D tensor map: one TMA per k-block (make_map_mn3)
  int passes;               // 1, or 2 halves of n / 2 columns (n = 512: the MMA's N is at most 256)
  int tmem_col;             // first accumulator column
  int relu, round_tf32;
  const float* bias;        // nullable
  const float* mask;        // nullable: keep the value where mask[row][col] > 0 (ReLU backward)
  long long ldmask;
  // the same test as one BIT per element: word [row][col / 32] of a (m, n / 32) uint32 matrix.  bits_out (forward):
  // bit j of the word = output column 32 w + j is positive; mask_bits (backward): keep the value where the bit is set.
  // A lane owns a row, so a 32-column chunk costs it one 4-byte load instead of 128 bytes of activations
  const uint32_t* mask_bits;
  uint32_t* bits_out;
};
struct ChainParams {
  int m, layers;
  ChainLayer L[3];
};
constexpr int CH_STAGE_B_BYTES = 256 * 128;
constexpr int CH_STAGE_BYTES = STAGE_A_BYTES + CH_STAGE_B_BYTES;
constexpr int CH_STAGES = 4;
constexpr int CH_SMEM_BYTES = CH_STAGES * CH_STAGE_BYTES + EPI_STAGE_BYTES + BAR_BYTES + 1024;

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
// D[tmem] (+)= A[tmem] B[smem]: A is 128 lanes x 8 columns of tf32 (raw fp32 bits) in tensor memory
__device__ __forceinline__ void tcgen05_mma_ts_tf32(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
               ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}

__global__ void __launch_bounds__(THREADS, 1)
chain_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b0,
                const __grid_constant__ CUtensorMap map_b1, const __grid_constant__ CUtensorMap map_b2,
                const __grid_constant__ CUtensorMap map_c0, const __grid_constant__ CUtensorMap map_c1,
                const __grid_constant__ CUtensorMap map_c2, const ChainParams p) {
  constexpr int BK = 32, UMMA_K = 8, MMAS_PER_STAGE = 4, MN_BOX = 32, MN_BOX_BYTES = 32 * 128;
  constexpr int MAX_PASSES = 4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* epi_smem = smem + CH_STAGES * CH_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_smem + EPI_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + CH_STAGES;
  uint64_t* acc_full = empty_bar + CH_STAGES;          // one per pass (each used once: a CTA owns one row block)
  uint64_t* a_ready = acc_full + MAX_PASSES;           // layer l's output is back in tensor memory as layer l+1's operand
  uint64_t* drained = a_ready + 3;                     // the first half of a two-pass layer has been read out
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained + 1);

  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const CUtensorMap* maps_b[3] = {&map_b0, &map_b1, &map_b2};
  const CUtensorMap* maps_c[3] = {&map_c0, &map_c1, &map_c2};
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    for (int l = 0; l < p.layers; ++l) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(maps_b[l]) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(maps_c[l]) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < CH_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int i = 0; i < MAX_PASSES; ++i) mbar_init(&acc_full[i], 1);
    for (int i = 0; i < 3; ++i) mbar_init(&a_ready[i], EPI_WARPS);
    mbar_init(drained, EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int row0 = blockIdx.x * BM;

  if (warp == 0) {
    // ===================== TMA producer: layer 1's rows and every layer's kernel, k-block by k-block =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int l = 0; l < p.layers; ++l) {
        const ChainLayer& L = p.L[l];
        const int nw = L.n / L.passes;
        for (int h = 0; h < L.passes; ++h) {
          for (int kb = 0; kb < L.k / BK; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * CH_STAGE_BYTES;
            uint8_t* sb = sa + STAGE_A_BYTES;
            mbar_expect_tx(&full_bar[stage], (l == 0 ? STAGE_A_BYTES : 0) + nw * 128);
            if (l == 0) tma_load_2d(sa, &map_a, &full_bar[stage], kb * BK, row0);
            if (L.b_mn3) {
              tma_load_3d(sb, maps_b[l], &full_bar[stage], 0, kb * BK, (h * nw) / MN_BOX);
            } else if (L.b_mn_major) {
              for (int j = 0; j < nw / MN_BOX; ++j)
                tma_load_2d(sb + j * MN_BOX_BYTES, maps_b[l], &full_bar[stage], h * nw + j * MN_BOX, kb * BK);
            } else {
              tma_load_2d(sb, maps_b[l], &full_bar[stage], kb * BK, h * nw);
            }
            if (++stage == CH_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int pass = 0;
      for (int l = 0; l < p.layers; ++l) {
        const ChainLayer& L = p.L[l];
        const int nw = L.n / L.passes;
        // D = f32, A / B = tf32, A K-major (or tensor memory), B as the layer says, N = nw, M = 128
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(L.b_mn_major) << 16) |
                               (uint32_t(nw >> 3) << 17) | (uint32_t(BM >> 4) << 24);
        const uint32_t b_lbo = L.b_mn_major ? MN_BOX_BYTES : 16;
        const uint32_t b_lt = L.b_mn_major ? 1u : 2u;
        const uint32_t b_sbo = b_lt == 1u ? 512u : 1024u;
        const uint32_t b_kstep = L.b_mn_major ? UMMA_K * 128 : 32;
        if (l > 0) {                                          // the previous layer's output is in tensor memory
          mbar_wait(&a_ready[l - 1], 0);
          tcgen05_fence_after();
        }
        for (int h = 0; h < L.passes; ++h, ++pass) {
          if (h > 0) {                                        // the second half reuses the first half's columns
            mbar_wait(drained, 0);
            tcgen05_fence_after();
          }
          const uint32_t tmem_d = tmem_base + L.tmem_col;
          for (int kb = 0; kb < L.k / BK; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tcgen05_fence_after();
            const uint32_t sa = smem_u32(smem + stage * CH_STAGE_BYTES);
            const uint32_t sb = sa + STAGE_A_BYTES;
#pragma unroll
            for (int k = 0; k < MMAS_PER_STAGE; ++k) {
              const uint64_t bdesc = make_desc(sb + k * b_kstep, b_lbo, b_sbo, b_lt);
              const uint32_t accum = (kb > 0 || k > 0) ? 1u : 0u;
              if (l == 0) {
                const uint64_t adesc = make_desc(sa + k * 32, 16, 1024, 2u);
                tcgen05_mma<KIND_TF32, 1>(tmem_d, adesc, bdesc, idesc, accum);
              } else {
                tcgen05_mma_ts_tf32(tmem_d, tmem_base + p.L[l - 1].tmem_col + kb * BK + k * UMMA_K, bdesc, idesc, accum);
              }
            }
            tcgen05_commit<1>(&empty_bar[stage]);
            if (++stage == CH_STAGES) { stage = 0; phase ^= 1; }
          }
          tcgen05_commit<1>(&acc_full[pass]);
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps): accumulator -> next operand in place, and -> global =====================
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;
    uint8_t* sbuf = epi_smem + (warp - 4) * 4096;
    const int row = row0 + q * 32 + lane;
    const bool row_ok = row < p.m;
    int pass = 0;
    for (int l = 0; l < p.layers; ++l) {
      const ChainLayer& L = p.L[l];
      const int nw = L.n / L.passes;
      const bool feeds_next = l + 1 < p.layers;
      for (int h = 0; h < L.passes; ++h, ++pass) {
        mbar_wait(&acc_full[pass], 0);
        tcgen05_fence_after();
        const int nch = nw / 64;                              // 32-column chunks of this warp's half
        for (int cb = 0; cb < nch; ++cb) {
          const int tcol = half * (nw / 2) + cb * 32;         // column inside the pass
          const int col0 = h * nw + tcol;                     // column of the layer's output
          const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(L.tmem_col + tcol);
          uint32_t v[32];
          __syncwarp();
          tmem_ld32(taddr, v);
          const float b_cur = L.bias ? __ldg(L.bias + col0 + lane) : 0.f;
          const float floor_v = L.relu ? 0.f : -INFINITY;
          float out[32];
#pragma unroll
          for (int j = 0; j < 32; ++j)
            out[j] = fmaxf(__uint_as_float(v[j]) + __shfl_sync(0xffffffffu, b_cur, j), floor_v);
          if (L.mask_bits) {
            const uint32_t word = row_ok ? __ldg(L.mask_bits + (long long)row * (L.n >> 5) + (col0 >> 5)) : 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) out[j] = ((word >> j) & 1u) ? out[j] : 0.f;
          } else if (L.mask) {
            if (row_ok) {
              const float* mrow = L.mask + (long long)row * L.ldmask + col0;
              if (((reinterpret_cast<uintptr_t>(mrow) | uintptr_t(L.ldmask * 4)) & 15) == 0) {     // 8 x 16 bytes per lane
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                  const float4 mk = __ldg(reinterpret_cast<const float4*>(mrow) + c);
                  out[4 * c] = mk.x > 0.f ? out[4 * c] : 0.f;         out[4 * c + 1] = mk.y > 0.f ? out[4 * c + 1] : 0.f;
                  out[4 * c + 2] = mk.z > 0.f ? out[4 * c + 2] : 0.f; out[4 * c + 3] = mk.w > 0.f ? out[4 * c + 3] : 0.f;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) out[j] = (__ldg(mrow + j) > 0.f) ? out[j] : 0.f;
              }
            }
          }
          if (L.round_tf32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) out[j] = rn_tf32_bits(out[j]);
          }
          if (L.bits_out && row_ok) {
            uint32_t word = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) word |= (out[j] > 0.f ? 1u : 0u) << j;
            L.bits_out[(long long)row * (L.n >> 5) + (col0 >> 5)] = word;
          }
          if (feeds_next) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(out[j]);
            tmem_st32(taddr, v);
          }
          if (lane == 0) tma_wait_group_read<0>();
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<float4*>(sbuf + lane * 128 + ((c ^ (lane & 7)) << 4)) =
                make_float4(out[4 * c], out[4 * c + 1], out[4 * c + 2], out[4 * c + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(maps_c[l], sbuf, col0, row0 + q * 32);
            tma_commit_group();
          }
        }
        if (feeds_next) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (feeds_next) mbar_arrive(&a_ready[l]);
          else if (L.passes == 2 && h == 0) mbar_arrive(drained);
        }
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

}  // namespace tc
}  // namespace cc

using namespace cc;

extern "C" {

// The planner behind cc_gemm_tc (host logic only: no device work): plan = {tile width, K split, CTAs per tile}.
// Candidates: (tile width, CTA pairing, K split); pairs only come as 256 x 256 tiles.
int cc_gemm_tc_plan(int precision, int m, int n, int k, int tile_n, int split_k, int* plan) {
  int p4[4];
  const int rc = cc_gemm_tc_plan_ex(precision, m, n, k, tile_n, split_k, p4);
  if (rc != CC_OK) return rc;
  CC_REQUIRE(plan, "cc_gemm_tc_plan: null plan");
  plan[0] = p4[0]; plan[1] = p4[1]; plan[2] = p4[2];
  return CC_OK;
}

// plan = {tile width, K split, CTAs per tile, hybrid stream-K (0 | 1)}.  Stream-K is only considered when the caller
// leaves the split to the planner (split_k == 0) and the dynamic tile scheduler is off; it comes with K split 1.
int cc_gemm_tc_plan_ex(int precision, int m, int n, int k, int tile_n, int split_k, int* plan) {
  CC_REQUIRE(plan && (precision == 1 || precision == 2) && m > 0 && n > 0 && k > 0, "cc_gemm_tc_plan: bad arguments");
  const int kblocks = ceil_div(k, precision == 2 ? 64 : 32);
  const int sms = sm_count();
  int bn = tile_n, split = split_k, ctas = 1, sk = 0;
  double best = -1.0;
  const int bns[3] = {256, 256, 128};
  const int cts[3] = {2, 1, 1};
  const bool sk_allowed = split_k == 0 && tc::g_stream_k != 0 && !tc::g_dynamic_tiles;
  for (int bi = 0; bi < 3; ++bi) {
    if (tile_n && bns[bi] != tile_n) continue;
    if (!tile_n && bns[bi] == 256 && n <= 128) continue;
    if (cts[bi] == 2 && tc::g_pair_mode == 0) continue;
    // small layers are latency-bound: single CTAs spread them over more SMs and skip the cluster handshakes
    if (cts[bi] == 2 && tc::g_pair_mode < 0 && 2.0 * m * n * double(k) < 2.0e10) continue;
    if (cts[bi] == 1 && tc::g_pair_mode == 1 && (tile_n == 0 || tile_n == 256) && n > 128) continue;
    const int smax = split_k > 0 ? split_k : (kblocks >= 16 ? (kblocks / 8 < 64 ? kblocks / 8 : 64) : 1);
    for (int s = (split_k > 0 ? split_k : 1); s <= smax; ++s) {
      const double e = tc::plan_eff(m, n, kblocks, bns[bi], s, sms, cts[bi]);
      if (e > best + 1e-9) { best = e; bn = bns[bi]; split = s; ctas = cts[bi]; sk = 0; }
    }
    // stream-K pays off on the big passes only (a small layer is a handful of tiles: latency-bound either way)
    if (sk_allowed && (tc::g_stream_k == 1 || 2.0 * m * n * double(k) >= 2.0e10)) {
      double e = tc::plan_eff_sk(m, n, kblocks, bns[bi], sms, cts[bi]);
      if (tc::g_stream_k == 1 && e > 0) e += 1.0;           // forced: beats every split plan of this shape
      if (e > best + 1e-9) { best = e; bn = bns[bi]; split = 1; ctas = cts[bi]; sk = 1; }
    }
  }
  plan[0] = bn; plan[1] = split; plan[2] = ctas; plan[3] = sk;
  return CC_OK;
}

// precision: 1 = tf32 (float operands), 2 = bf16 (__nv_bfloat16 operands; C, bias, mask stay float).
// split_k: 0 = choose (tile width and split) automatically, >= 1 = as given (tile_n: 0 auto | 128 | 256).
int cc_gemm_tc(int precision, int transa, int transb, int m, int n, int k, const void* a, int64_t lda, const void* b,
               int64_t ldb, float* c, int64_t ldc, const float* bias, int relu, const float* mask, int64_t ldmask,
               int accumulate, int split_k, int tile_n, int round_tf32, void* stream) {
  CC_NVTX("cc_gemm_tc");
  CC_REQUIRE(a && b && c, "cc_gemm_tc: null pointer");
  CC_REQUIRE(precision == 1 || precision == 2, "cc_gemm_tc: precision must be 1 (tf32) or 2 (bf16)");
  CC_REQUIRE(m >= 0 && n >= 0 && k > 0, "cc_gemm_tc: bad sizes m=%d n=%d k=%d", m, n, k);
  CC_REQUIRE(tile_n == 0 || tile_n == 128 || tile_n == 256, "cc_gemm_tc: tile_n must be 0, 128 or 256");
  if (m == 0 || n == 0) return CC_OK;
  cudaStream_t st = as_stream(stream);
  int plan[4];
  cc_gemm_tc_plan_ex(precision, m, n, k, tile_n, split_k, plan);
  const int bn = plan[0], split = plan[1], ctas = plan[2], sk = plan[3];
  const bool nonlinear = bias || relu || mask || round_tf32;
  const bool two_pass = (split > 1 || sk) && nonlinear;
  CC_REQUIRE(!(two_pass && accumulate), "cc_gemm_tc: accumulate with a split-K non-linear epilogue is not supported");
  tc::Params p{};
  p.m = m; p.n = n; p.k = k; p.n_store = n;
  p.bias = two_pass ? nullptr : bias; p.mask = two_pass ? nullptr : mask; p.ldmask = ldmask;
  p.relu = two_pass ? 0 : relu; p.round_tf32 = two_pass ? 0 : round_tf32;
  p.split_k = split;
  p.sk_tiles = sk ? -1 : 0;              // -1: launch_bn sizes the stream-K part for the units it can actually run
  p.reduce_add = (accumulate || split > 1) ? 1 : 0;
  if (split > 1 && !accumulate)
    CC_CHECK_CUDA(cudaMemset2DAsync(c, size_t(ldc) * 4, 0, size_t(n) * 4, m, st));
  tc::Problem pr{transa, transb, m, n, k, a, lda, b, ldb, c, ldc, precision == 2 ? tc::KIND_BF16 : tc::KIND_TF32};
  int rc = precision == 2 ? tc::launch<tc::KIND_BF16, tc::EPI_STORE>(pr, p, bn, ctas, st)
                          : tc::launch<tc::KIND_TF32, tc::EPI_STORE>(pr, p, bn, ctas, st);
  if (rc != CC_OK) return rc;
  if (two_pass) {
    const long long total = (long long)m * n;
    tc::post_epilogue_kernel<<<(unsigned)ceil_div<long long>(total, 256LL), 256, 0, st>>>(c, ldc, m, n, bias, relu, mask,
                                                                                         ldmask, round_tf32);
    CC_CHECK_LAUNCH();
  }
  return CC_OK;
}

// Fused decoder output layer + sigmoid-BCE:  z = A[M,K] W[K,N] + bias;  loss partials and
// dlogits = (sigmoid(z) - y)/count written to dz[M][lddz] (columns [N, lddz) zeroed).
// loss_partial: float64 [cc_gemm_bce_partial_count(m, lddz)]  (sum it with cc_loss_finalize).
// dz == NULL: loss only (evaluation) -- the partials are the same, nothing else is written; lddz still sizes the
// partial array, dbias must be NULL and dz_bf16 0.
int cc_gemm_bce_tc(int precision, int m, int n, int k, const void* a, int64_t lda, const void* w, int64_t ldw,
                   const float* bias, const uint32_t* ybits, int64_t ywords, double count, void* dz, int64_t lddz,
                   double* loss_partial, float* dbias, int round_tf32, int dz_bf16, void* stream) {
  return cc_gemm_bce_tc_ex(precision, m, n, k, a, lda, w, ldw, bias, ybits, ywords, count, dz, lddz, loss_partial, dbias,
                           round_tf32, dz_bf16, nullptr, stream);
}

// acc_partial (nullable, float64, same size and layout as loss_partial): per-(tile, warp) counts of the cells whose
// rounded probability equals the label, i.e. Keras' binary_accuracy numerator (metrics=['accuracy'], train.py:87).
int cc_gemm_bce_tc_ex(int precision, int m, int n, int k, const void* a, int64_t lda, const void* w, int64_t ldw,
                      const float* bias, const uint32_t* ybits, int64_t ywords, double count, void* dz, int64_t lddz,
                      double* loss_partial, float* dbias, int round_tf32, int dz_bf16, double* acc_partial, void* stream) {
  CC_NVTX("cc_gemm_bce_tc");
  CC_REQUIRE(a && w && bias && ybits && loss_partial, "cc_gemm_bce_tc: null pointer");
  CC_REQUIRE(dz || (!dbias && !dz_bf16), "cc_gemm_bce_tc: loss only (dz == NULL) takes no dbias and no bf16 dlogits");
  CC_REQUIRE(precision == 1 || precision == 2, "cc_gemm_bce_tc: precision must be 1 (tf32) or 2 (bf16)");
  CC_REQUIRE(m > 0 && n > 0 && k > 0 && count > 0, "cc_gemm_bce_tc: bad sizes");
  CC_REQUIRE(lddz % 32 == 0 && lddz >= n && ywords * 32 >= lddz,
             "cc_gemm_bce_tc: lddz must be a multiple of 32 >= n and ywords*32 >= lddz");
  tc::Params p{};
  p.m = m; p.n = n; p.k = k; p.n_store = int(lddz);
  p.bias = bias; p.split_k = 1; p.round_tf32 = round_tf32;
  p.ybits = ybits; p.ywords = ywords; p.inv_count = float(1.0 / count); p.loss_partial = loss_partial;
  p.dbias = dbias;
  p.acc_partial = acc_partial;
  if (dbias) CC_CHECK_CUDA(cudaMemsetAsync(dbias, 0, size_t(n) * sizeof(float), as_stream(stream)));
  tc::Problem pr{0, 0, m, n, k, a, lda, w, ldw, static_cast<float*>(dz), lddz, precision == 2 ? tc::KIND_BF16 : tc::KIND_TF32};
  const int ctas = tc::g_pair_mode == 0 ? 1 : 2;
  if (!dz) {
    if (acc_partial) {
      if (precision == 2) return tc::launch<tc::KIND_BF16, tc::EPI_BCE_LOSS_ACC>(pr, p, 256, ctas, as_stream(stream));
      return tc::launch<tc::KIND_TF32, tc::EPI_BCE_LOSS_ACC>(pr, p, 256, ctas, as_stream(stream));
    }
    if (precision == 2) return tc::launch<tc::KIND_BF16, tc::EPI_BCE_LOSS>(pr, p, 256, ctas, as_stream(stream));
    return tc::launch<tc::KIND_TF32, tc::EPI_BCE_LOSS>(pr, p, 256, ctas, as_stream(stream));
  }
  if (dz_bf16) {
    CC_REQUIRE(precision == 2, "cc_gemm_bce_tc: bf16 dlogits come with bf16 operands (precision 2)");
    p.round_tf32 = 0;
    if (acc_partial) return tc::launch<tc::KIND_BF16, tc::EPI_BCE16_ACC>(pr, p, 256, ctas, as_stream(stream));
    return tc::launch<tc::KIND_BF16, tc::EPI_BCE16>(pr, p, 256, ctas, as_stream(stream));
  }
  if (acc_partial) {
    if (precision == 2) return tc::launch<tc::KIND_BF16, tc::EPI_BCE_ACC>(pr, p, 256, ctas, as_stream(stream));
    return tc::launch<tc::KIND_TF32, tc::EPI_BCE_ACC>(pr, p, 256, ctas, as_stream(stream));
  }
  if (precision == 2) return tc::launch<tc::KIND_BF16, tc::EPI_BCE>(pr, p, 256, ctas, as_stream(stream));
  return tc::launch<tc::KIND_TF32, tc::EPI_BCE>(pr, p, 256, ctas, as_stream(stream));
}

// one float64 per (128-row block, 256-column tile, epilogue warp); sized for the CTA-pair tiling (256-row
// tiles, both CTAs) -- entries a launch does not cover stay untouched (the caller zero-initialises once)
int64_t cc_gemm_bce_partial_count(int m, int lddz) {
  return int64_t(ceil_div(m, 2 * tc::BM)) * 2 * ceil_div(lddz, 256) * tc::EPI_WARPS;
}

// Co-occurrence counts cnt = X^T X on the tensor cores (reference src/non_ml/utils.py:82-84): the cubes of a chunk
// are expanded to a K-major byte matrix X^T [C][chunk] and contracted with tcgen05.mma kind::i8 (0/1 bytes, int32
// accumulators -> exact), upper-triangle tiles only, each off-diagonal tile mirrored by the epilogue.
static const int64_t kCountChunk = 32768;      // cubes per pass (the byte matrix is C x chunk)

int64_t cc_cooc_tc_chunk_cubes(int64_t num_cubes) {
  const int64_t k = num_cubes < kCountChunk ? num_cubes : kCountChunk;
  return (k + 127) / 128 * 128;
}
int64_t cc_cooc_tc_workspace_bytes(int64_t num_cubes, int32_t num_cards) {
  return cc_cooc_tc_chunk_cubes(num_cubes) * int64_t(num_cards) + 1024;
}

int cc_cooc_count_tc(const int64_t* indptr, const int32_t* indices, int64_t num_cubes, int32_t num_cards,
                     void* workspace, int64_t workspace_bytes, int32_t* counts, int64_t ldc, int accumulate,
                     int32_t* bad, void* stream) {
  CC_NVTX("cc_cooc_count_tc");
  CC_REQUIRE(indptr && indices && workspace && counts, "cc_cooc_count_tc: null pointer");
  CC_REQUIRE(num_cubes >= 0 && num_cards > 0 && ldc >= num_cards, "cc_cooc_count_tc: bad sizes");
  CC_REQUIRE(ldc % 4 == 0 && (reinterpret_cast<uintptr_t>(counts) & 15) == 0,
             "cc_cooc_count_tc: counts needs a 16-byte aligned base and ldc %% 4 == 0 (ldc=%lld)", (long long)ldc);
  CC_REQUIRE(workspace_bytes >= cc_cooc_tc_workspace_bytes(num_cubes, num_cards), "cc_cooc_count_tc: workspace too small");
  cudaStream_t st = as_stream(stream);
  if (num_cubes == 0) {
    if (!accumulate) CC_CHECK_CUDA(cudaMemset2DAsync(counts, size_t(ldc) * 4, 0, size_t(num_cards) * 4, num_cards, st));
    return CC_OK;
  }
  bool add = accumulate != 0;           // the first pass of a fresh build stores (every element is covered), later ones add
  uint8_t* xt = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~uintptr_t(1023));
  const int64_t ldx = cc_cooc_tc_chunk_cubes(num_cubes);
  for (int64_t k0 = 0; k0 < num_cubes; k0 += kCountChunk) {
    const int chunk = int(num_cubes - k0 < kCountChunk ? num_cubes - k0 : kCountChunk);
    const int kpad = (chunk + 127) / 128 * 128;
    CC_CHECK_CUDA(cudaMemset2DAsync(xt, size_t(ldx), 0, size_t(kpad), num_cards, st));
    const int wpb = 8;
    tc::expand_cubes_u8_kernel<<<ceil_div(chunk, wpb), wpb * 32, 0, st>>>(indptr, indices, k0, chunk, num_cards, xt, ldx, bad);
    CC_CHECK_LAUNCH();
    tc::Params p{};
    p.m = num_cards; p.n = num_cards; p.k = kpad; p.n_store = num_cards;
    p.split_k = 1; p.symmetric = 1;
    {
      const int n = ceil_div(num_cards, 256);
      int g = 8;                                            // 8 row blocks x 256 cards x <= 32 KB = <= 64 MB of A in L2
      while (ceil_div(n, g) > 71) ++g;
      p.band_rows = g;
      int acc = 0, b = 0;
      for (int r0 = 0; r0 < n; r0 += g, ++b) {
        p.band_start[b] = acc;
        const int rows = (g < n - r0) ? g : n - r0;
        acc += rows * (rows + 1) / 2 + (n - r0 - rows) * rows;
      }
      p.band_start[b] = acc;
      for (int i = b + 1; i < 72; ++i) p.band_start[i] = 0x7fffffff;
    }
    p.reduce_add = add ? 1 : 0;
    add = true;
    p.count_out = counts; p.ldcount = ldc;
    tc::Problem pr{0, 1, num_cards, num_cards, kpad, xt, ldx, xt, ldx, reinterpret_cast<float*>(counts), ldc, tc::KIND_U8};
    const int rc = tc::launch<tc::KIND_U8, tc::EPI_COUNT>(pr, p, 256, 2, st);
    if (rc != CC_OK) return rc;
  }
  return CC_OK;
}

// Up to three consecutive small Dense layers in one launch (see chain_tc_kernel): widths = {k0, n1, ..., n_layers};
// layer l computes out_l[m][n_l] = epi(in_l W_l) with in_1 = a and in_{l+1} = out_l.  w_is_kn[l] = 1: W_l is the Keras
// kernel [K][N] (forward), 0: it is [N][K] (the transposed use of a kernel in backward).  bias[l] / mask[l] nullable;
// relu applies to every layer that has a bias (forward), the mask test (mask > 0) is ReLU's backward; mask_bits /
// bits_out carry the same test as one bit per element ((m, n / 32) uint32 matrices, see ChainLayer).
int cc_chain_tc(int m, int layers, const int32_t* widths, const float* a, int64_t lda, const float* const* w,
                const int64_t* ldw, const int32_t* w_is_kn, const float* const* bias, const float* const* mask,
                const int64_t* ldmask, const uint32_t* const* mask_bits, uint32_t* const* bits_out, int relu,
                float* const* out, const int64_t* ldout, int round_tf32, void* stream) {
  CC_NVTX("cc_chain_tc");
  CC_REQUIRE(m > 0 && layers >= 1 && layers <= 3, "cc_chain_tc: 1..3 layers (got %d) and m > 0", layers);
  CC_REQUIRE(widths && a && w && ldw && w_is_kn && out && ldout, "cc_chain_tc: null argument");
  tc::ChainParams p{};
  p.m = m; p.layers = layers;
  int total = 0;
  for (int l = 0; l < layers; ++l) {
    const int k = widths[l], n = widths[l + 1];
    CC_REQUIRE(k % 32 == 0 && k >= 32 && k <= 512 && n % 64 == 0 && n >= 64 && n <= 512,
               "cc_chain_tc: layer %d is %d -> %d (k must be a multiple of 32, n of 64, both <= 512)", l, k, n);
    CC_REQUIRE(n <= 256 || l == layers - 1, "cc_chain_tc: only the last layer may be 512 wide");
    CC_REQUIRE((reinterpret_cast<uintptr_t>(w[l]) & 15) == 0 && (reinterpret_cast<uintptr_t>(out[l]) & 15) == 0 &&
                   (ldw[l] * 4) % 16 == 0 && (ldout[l] * 4) % 16 == 0,
               "cc_chain_tc: layer %d: kernels and outputs must be 16-byte aligned with leading dimensions % 4 == 0", l);
    tc::ChainLayer& L = p.L[l];
    L.n = n; L.k = k; L.b_mn_major = w_is_kn[l] ? 1 : 0; L.passes = n > 256 ? 2 : 1;
    L.relu = (relu && bias && bias[l]) ? 1 : 0; L.round_tf32 = round_tf32;
    L.bias = bias ? bias[l] : nullptr;
    L.mask = mask ? mask[l] : nullptr;
    L.ldmask = (mask && mask[l] && ldmask) ? ldmask[l] : 0;
    L.mask_bits = mask_bits ? mask_bits[l] : nullptr;
    L.bits_out = bits_out ? bits_out[l] : nullptr;
    total += n;
  }
  CC_REQUIRE((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (lda * 4) % 16 == 0, "cc_chain_tc: a must be 16-byte aligned, lda % 4 == 0");
  // tensor-memory columns (512 per SM): consecutive accumulators when they fit; otherwise (64 -> 128 -> 256 -> 512) the
  // last layer's two 256-column halves reuse the columns of the first accumulator, which is dead by then
  if (total <= 512) {
    int c = 0;
    for (int l = 0; l < layers; ++l) { p.L[l].tmem_col = c; c += p.L[l].n / p.L[l].passes; }   // (two halves share their columns)
  } else {
    CC_REQUIRE(layers == 3 && p.L[2].passes == 2 && p.L[0].n <= 256 && p.L[1].n <= 256,
               "cc_chain_tc: accumulators of %d columns do not fit the 512 columns of tensor memory", total);
    p.L[0].tmem_col = 0; p.L[1].tmem_col = 256; p.L[2].tmem_col = 0;
  }
  CUtensorMap map_a, map_b[3], map_c[3];
  int rc = tc::make_map(&map_a, a, 4, tc::MAP_F32, m, widths[0], lda, tc::BM, false);
  if (rc != CC_OK) return rc;
  for (int l = 0; l < 3; ++l) {
    const int ll = l < layers ? l : layers - 1;               // unused slots repeat the last layer's maps
    tc::ChainLayer& L = p.L[ll];
    const int nw = L.n / L.passes;
    if (l == ll) L.b_mn3 = (L.b_mn_major && tc::g_mn3) ? 1 : 0;
    if (L.b_mn3 && tc::make_map_mn3(&map_b[l], w[ll], L.k, L.n, ldw[ll], nw / 32) != CC_OK) {
      CC_REQUIRE(l == ll, "cc_chain_tc: tensor map of a repeated slot failed");
      L.b_mn3 = 0;                                            // (driver refused the 3-D form: 2-D boxes)
    }
    if (L.b_mn3)           { rc = CC_OK; if (l == ll) ++tc::g_mn3_used; }
    else if (L.b_mn_major) rc = tc::make_map(&map_b[l], w[ll], 4, tc::MAP_F32, L.k, L.n, ldw[ll], 32, true);
    else                   rc = tc::make_map(&map_b[l], w[ll], 4, tc::MAP_F32, L.n, L.k, ldw[ll], nw, false);
    if (rc != CC_OK) return rc;
    rc = tc::make_map(&map_c[l], out[ll], 4, tc::MAP_F32, m, L.n, ldout[ll], 32, false);
    if (rc != CC_OK) return rc;
  }
  static std::mutex mu;
  static bool attr_done[64] = {false};
  int dev = 0;
  CC_CHECK_CUDA(cudaGetDevice(&dev));
  CC_REQUIRE(dev >= 0 && dev < 64, "cc_chain_tc: device ordinal %d out of range", dev);
  {
    std::lock_guard<std::mutex> lk(mu);
    if (!attr_done[dev]) {
      CC_CHECK_CUDA(cudaFuncSetAttribute(tc::chain_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::CH_SMEM_BYTES));
      attr_done[dev] = true;
    }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(unsigned((m + tc::BM - 1) / tc::BM));
  cfg.blockDim = dim3(tc::THREADS);
  cfg.dynamicSmemBytes = tc::CH_SMEM_BYTES;
  cfg.stream = as_stream(stream);
  cudaLaunchAttribute at[1];
  int na = 0;
  if (tc::g_pdl) {
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = at; cfg.numAttrs = na;
  CC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, tc::chain_tc_kernel, map_a, map_b[0], map_b[1], map_b[2], map_c[0], map_c[1], map_c[2], p));
  CC_CHECK_LAUNCH();
  return CC_OK;
}

// number of MN-major tf32 operands that went through a 3-D tensor map since the library was loaded (0 after MN-major
// launches means the driver refused the 3-D form and the 2-D boxes were used)
int64_t cc_gemm_tc_mn3_count(void) { return int64_t(tc::g_mn3_used.load()); }

// Declares [base, base + bytes) readable in full for as long as GEMMs are launched on operands inside it (bytes = 0
// forgets the range that starts at base).  See readable_range: it lets unpadded MN-major tf32 operands inside the range
// take the single-TMA 3-D form, whose last column group of a row reads up to 124 bytes past the row's end.
int cc_gemm_tc_register_readable(const void* base, int64_t bytes) {
  CC_REQUIRE(base != nullptr && bytes >= 0, "cc_gemm_tc_register_readable: null base or negative size");
  std::lock_guard<std::mutex> lk(tc::g_readable_mu);
  const uintptr_t lo = reinterpret_cast<uintptr_t>(base);
  int slot = -1;
  for (int i = 0; i < tc::g_readable_n; ++i) if (tc::g_readable[i][0] == lo) slot = i;
  if (bytes == 0) {
    if (slot >= 0) { tc::g_readable[slot][0] = tc::g_readable[tc::g_readable_n - 1][0]; tc::g_readable[slot][1] = tc::g_readable[tc::g_readable_n - 1][1]; --tc::g_readable_n; }
    return CC_OK;
  }
  if (slot < 0) {
    if (tc::g_readable_n == 32) { tc::g_readable_n = 0; }     // (a table of the most recent ranges: start over)
    slot = tc::g_readable_n++;
  }
  tc::g_readable[slot][0] = lo; tc::g_readable[slot][1] = lo + uintptr_t(bytes);
  return CC_OK;
}

int cc_gemm_tc_set_pdl(int on) {
  tc::g_pdl = on ? 1 : 0;
  return CC_OK;
}

int cc_gemm_tc_set_dynamic_tiles(int on) {
  tc::g_dynamic_tiles = on ? 1 : 0;
  return CC_OK;
}

int cc_gemm_tc_set_stream_k(int mode) {
  CC_REQUIRE(mode >= -1 && mode <= 1, "cc_gemm_tc_set_stream_k: mode must be -1 (auto), 0 (off) or 1 (on)");
  tc::g_stream_k = mode;
  return CC_OK;
}

int cc_gemm_tc_set_pair_mode(int mode) {
  CC_REQUIRE(mode >= -1 && mode <= 1, "cc_gemm_tc_set_pair_mode: mode must be -1 (auto), 0 (off) or 1 (on)");
  tc::g_pair_mode = mode;
  return CC_OK;
}

}  // extern "C"
