// Plane-native tcgen05 dense pipeline: fp32-accurate GEMMs whose operands AND results live in HBM as
// pre-split hi/lo planes (plane_fmt.cuh), so no conversion pass sits between the layers of a subnetwork.
//
// Two plane formats share one kernel template:
//   FMT_F16  (default)  hi = fp16(T), lo' = fp16((T - hi) 2^11); 2 B / value, k-block = 64 columns;
//                       tcgen05.mma.kind::f16, C = sum a_hi b_hi + 2^-11 sum (a_hi b_lo' + a_lo' b_hi)
//   FMT_TF32 (fallback) hi = rna_tf32(T), lo = rna_tf32(T - hi); 4 B / value, k-block = 32 columns;
//                       tcgen05.mma.kind::tf32, C = sum a_hi b_hi + sum (a_hi b_lo + a_lo b_hi)
// Both carry 22 significant bits per value and drop only the lo*lo term (2^-22 relative).
//
// Planes of T[rows, cols] are k-block-major  plane[cols/BK][rows][BK]  (one 128 B row per (k-block, row)),
// zero padded in cols, followed by sign bits  bits[cols/32][rows]  (the ReLU mask of the backward pass costs
// 1/32..1/16 of a plane instead of a 4 B/element read).  One layout serves every GEMM of training because
// tcgen05 takes either operand K-major or MN-major straight from shared memory:
//     K  = cols of T : box {BK, 128 rows, 1 kb}        -> K-major  [128 rows][BK]           SWIZZLE_128B
//     K  = rows of T : box {BK, BK rows, 128/BK kb}    -> MN-major [128/BK][BK k][BK mn]    SWIZZLE_128B (f16)
//                                                                                           SWIZZLE_128B_ATOM_32B (tf32)
//   all boxes are 16 KiB.
//     fwd  Y = X W       A = Xp  K-major (K=in)    B = Wp  MN-major (N=out, K=in)
//     dX   = dZ W^T      A = dZp K-major (K=out)   B = Wp  K-major  (N=in,  K=out)
//     dW   = X^T dZ      A = Xp  MN-major (M=in)   B = dZp MN-major (N=out), K = batch
//   -> no transposed copies, and the epilogue of one GEMM writes the planes the
//   next one reads (bias+ReLU for fwd, ReLU mask + column sums for dX).
//
// The tensor core truncates its fp32 accumulator on every add, so hi*hi partial sums stay in TMEM for
// 128 K only and are then added in registers with RN (profiles/r1a_accuracy_probe_*.txt,
// profiles/r2a_proto_f16.txt); cross terms use their own accumulator.
//
// Kernel: persistent, one CTA per SM, 576 threads, warp-specialised, grouped (up to 8 GEMMs per launch)
//   warp 0    TMA producer (3-stage ring, 64 KiB per stage: A_hi A_lo B_hi B_lo)
//   warp 1    MMA issuer (elected lane; per K step one N=256 MMA a_hi x [b_hi|b_lo] + one N=128 MMA a_lo x b_hi)
//   warps 2-17 epilogue (TMEM lane quadrant = warp % 4, column group = (warp-2)/4, 32 accumulators each):
//             tcgen05.ld -> registers (bias/ReLU/dropout + sign bits | sign-bit mask + column sums) -> hi/lo split
//             -> planes out: the warp's 2 KB smem slab + one TMA store per plane ([32 rows][32 columns] box);
//                dense fp32 out (logits, dW partials): per-warp swizzled smem transpose -> full-sector stores
//
// Reference arithmetic replaced: tf.layers.dense and its gradients,
//   adanet/examples/simple_dnn.py:72-86,103-110.
#include <cuda.h>
#include <cudaTypedefs.h>

#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "dense_simt.cuh"
#include "planes.cuh"

namespace adn {
namespace pl {

static constexpr int BM = 128, BN = 128;
static constexpr int STAGES = 3;
static constexpr int TILE_BYTES = 128 * 128;          // 16 KiB: 128 rows x one 128 B k-block row
static constexpr int STAGE_BYTES = 4 * TILE_BYTES;    // A_hi A_lo B_hi B_lo
// 16 epilogue warps x 32 columns (TMEM lane quadrant = warp % 4, column group = (warp-2)/4): the short-K layer
// waves are bound by epilogue latency per warp, so thread-level parallelism is what helps; each warp stages
// 32x16 floats (2 KB) at a time to stay inside the 32 KB left beside the 3-stage ring.
static constexpr int EPI_WARPS = 16;
static constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
static constexpr int EPI_STAGE_FLOATS = 32 * 16;
static constexpr int EPI_BYTES = EPI_WARPS * EPI_STAGE_FLOATS * 4;
static constexpr int BAR_BYTES = 256;
static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + BAR_BYTES;
static constexpr int TMEM_COLS = 512;                 // two chunk buffers of [H: 128 | S: 128] columns
static constexpr int MAX_SPLITS = 64;

template <int FMT> struct Fmt;
template <> struct Fmt<FMT_TF32> {
  static constexpr int BK = 32;          // columns per k-block (128 B)
  static constexpr int CHUNK = 4;        // k-blocks per TMEM accumulation chunk (K = 128)
  static constexpr uint32_t MN_STEP = 1024u >> 4;   // descriptor address advance per MMA, MN-major operand (8 k rows)
  static constexpr uint32_t MN_LBO = 4096u >> 4;    // next 32-wide mn block
  static constexpr uint32_t MN_HI = (uint32_t)(512 >> 4) | (1u << 14) | (1u << 29);   // SBO 512, SWIZZLE_128B_BASE32B
  static constexpr uint32_t IDESC_AB = (2u << 7) | (2u << 10);                        // a = b = TF32
};
template <> struct Fmt<FMT_F16> {
  static constexpr int BK = 64;
  static constexpr int CHUNK = 2;        // K = 128
  static constexpr uint32_t MN_STEP = 2048u >> 4;   // 16 k rows
  static constexpr uint32_t MN_LBO = 8192u >> 4;    // next 64-wide mn block
  static constexpr uint32_t MN_HI = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);  // SBO 1024, SWIZZLE_128B
  static constexpr uint32_t IDESC_AB = 0u;                                            // a = b = F16
};

enum { EPI_BIAS_ACT = 0, EPI_MASK = 1, EPI_PARTIAL = 2 };

struct GemmParams {
  int M, N;
  int tiles_m, tiles_n, splits;
  int tiles;             // tiles_m * tiles_n
  float inv_tiles, inv_tiles_n;   // reciprocals for the division-free item decode (counts stay far below 2^21)
  int total_kb;          // k-blocks over the whole K
  int kb_per_split;
  int a_mn, b_mn;        // operand majorness (0 = K-major box, 1 = MN-major box)
  int out_planes;        // 1: result written as split planes (out / out_lo / out_bits), 0: dense fp32
  // output: dense row-major (ldc) / split-K partial [split][M][N], or planes
  void* out;             // dense base | hi plane base
  void* out_lo;          // lo plane base (OUT_PLANES)
  int ldc;
  int out_nb32;          // planes: 32-column blocks of the (padded) output tensor
  int out_tma;           // planes (fp16): the tile is written through shared memory with TMA stores (Problem::o_hi / o_lo)
  const float* bias;     // EPI_BIAS_ACT (nullable)
  int act;
  uint32_t* out_bits;    // planes + EPI_BIAS_ACT: sign bits of the output
  const uint32_t* mask_bits;  // EPI_MASK (nullable): sign bits of a [M, N] tensor; out = bit ? out : 0
  float* colsum_part;    // EPI_MASK (nullable): [ceil(M/32)][colsum_ld] per-32-row column sums of out
  int colsum_ld;
  float out_mul;         // EPI_MASK / EPI_PARTIAL: result multiplied by this (un-scaling of gradient planes, 1/(1-rate) of dropout)
  unsigned int* ovf;     // sticky overflow word (fp16 planes)
  // EPI_BIAS_ACT with planes out: tf.layers.dropout on the output (drop_thresh 0 = none)
  uint32_t drop_thresh;  // keep iff hash >= thresh (= rate * 2^32)
  uint32_t drop_key0;    // seed * 0x9E3779B1 + layer * 0x85EBCA77 + 0x27D4EB2F  (the step term is added on the device)
  float drop_scale;      // 1 / (1 - rate)
  const int64_t* drop_step;
};

// ---------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded spin: a broken pipeline traps (CUDA error) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    if ((it & 1023u) == 1023u) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) __trap();   // ~2 s at 2 GHz
    }
  }
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// shared -> global tile store (bulk async-group completion); coordinates past the tensor bounds are clipped
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 | [32,46) SBO >> 4 | [46,48) version = 1 | [61,64) layout type
//   K-major  tile [128 rows][128 B of k], SWIZZLE_128B (type 2): SBO = 1024 (8 rows x 128 B), LBO unused (=1);
//            next MMA (K = 8 tf32 / 16 f16): +32 B
//   MN-major tile [128/BK mn-blocks][BK k][BK mn] (each k row 128 B):
//     f16 : SWIZZLE_128B (type 2), atom = 64 mn x 8 k rows: LBO = 8192 (next 64-wide mn block), SBO = 1024
//           (next 8 k rows); next MMA (16 k rows): +2048 B
//     tf32: 32-bit MN-major operands must use the 32 B-granular 128 B swizzle SWIZZLE_128B_BASE32B (type 1, TMA
//           CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B; atom = 32 mn x 4 k rows): LBO = 4096, SBO = 512; next MMA
//           (8 k rows): +1024 B
static constexpr uint32_t K_MAJOR_HI = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
template <int FMT>
__device__ __forceinline__ uint32_t desc_hi_word(int mn_major) { return mn_major ? Fmt<FMT>::MN_HI : K_MAJOR_HI; }
template <int FMT>
__device__ __forceinline__ uint32_t desc_lo_word(uint32_t smem_addr, int mn_major) {
  return ((smem_addr & 0x3FFFFu) >> 4) | ((mn_major ? Fmt<FMT>::MN_LBO : 1u) << 16);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6)=1, a format [7,10), b format [10,13)
// (0 = F16, 2 = TF32), a_major [15], b_major [16] (0 = K, 1 = MN), n_dim=N>>3 [17,23), m_dim=M>>4 [24,29).
template <int FMT>
__device__ __forceinline__ uint32_t make_idesc(int m, int n, int a_mn, int b_mn) {
  return (1u << 4) | Fmt<FMT>::IDESC_AB | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
template <int FMT>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint32_t da_lo, uint32_t db_lo, uint32_t da_hi, uint32_t db_hi,
                                     uint32_t idesc, uint32_t accum) {
  if (FMT == FMT_F16) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
        ::"r"(tmem_d), "r"(da_lo), "r"(db_lo), "r"(da_hi), "r"(db_hi), "r"(idesc), "r"(accum)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
        ::"r"(tmem_d), "r"(da_lo), "r"(db_lo), "r"(da_hi), "r"(db_hi), "r"(idesc), "r"(accum)
        : "memory");
  }
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

// work item -> (tile_m, tile_n, split).  n fastest so concurrently resident CTAs share A tiles through L2 (A is the
// big operand of the long-K layers).
struct Item {
  int m0, n0, kb0, nkb, split;
};
// q = n / d for 0 <= n < 2^21 with inv = 1.0f / d: (n + 0.5) / d is never within 1/(2d) of an integer, far more than the
// fp32 error of the product, so the truncation is exact.  (An integer division is ~20 instructions; every one of the 18
// warps of a CTA decodes every work item, and on the thin-K layer waves that was a quarter of the stall samples.)
__device__ __forceinline__ int fast_div(int n, float inv) { return (int)(((float)n + 0.5f) * inv); }

__device__ __forceinline__ Item decode_item(const GemmParams& g, int item) {
  Item it;
  it.split = (g.splits == 1) ? 0 : fast_div(item, g.inv_tiles);
  const int t = item - it.split * g.tiles;
  const int tm = (g.tiles_n == 1) ? t : fast_div(t, g.inv_tiles_n);
  it.m0 = tm * BM;
  it.n0 = (t - tm * g.tiles_n) * BN;
  it.kb0 = it.split * g.kb_per_split;
  it.nkb = min(g.total_kb, it.kb0 + g.kb_per_split) - it.kb0;
  return it;
}

__device__ __forceinline__ uint32_t pack_h2(__half a, __half b) {
  return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}

// One 32-row x 32-column slice of a tile: lane = row holds its 32 accumulators a[0..31] (columns
// cbase..cbase+31).  Applies bias/ReLU (+ sign bits) or the sign-bit ReLU mask in the register layout,
// transposes through `stage` (16 B chunks XOR-swizzled by row: conflict-free both ways) and writes with
// lane = 4-column group of 8 rows, so every global access covers whole 32 B sectors.
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t (&w)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
               "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}

// split 32 values of one row into the two planes and write them with 256-bit stores (TF32 planes, and fp16 planes whose
// buffers are not 128 B aligned or hold an odd number of 32-column blocks; other fp16 planes take store_slice_tma_hi / _lo)
template <int FMT>
__device__ __forceinline__ void store_row32_planes(const GemmParams& g, const float* a, int my_row, int cbase) {
  constexpr int BK = Fmt<FMT>::BK;
  const size_t poff = ((size_t)(cbase / BK) * g.M + my_row) * BK + (cbase % BK);
  if (FMT == FMT_F16) {
    uint32_t hw[16], lw[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const __half2 h2 = __floats2half2_rn(a[2 * q], a[2 * q + 1]);
      const float2 hf = __half22float2(h2);
      const __half2 l2 = __floats2half2_rn((a[2 * q] - hf.x) * 2048.0f, (a[2 * q + 1] - hf.y) * 2048.0f);
      hw[q] = *reinterpret_cast<const uint32_t*>(&h2);
      lw[q] = *reinterpret_cast<const uint32_t*>(&l2);
    }
    __half* hp = reinterpret_cast<__half*>(g.out) + poff;
    __half* lp = reinterpret_cast<__half*>(g.out_lo) + poff;
    st_global_v8(hp, reinterpret_cast<const uint32_t(&)[8]>(hw[0]));
    st_global_v8(hp + 16, reinterpret_cast<const uint32_t(&)[8]>(hw[8]));
    st_global_v8(lp, reinterpret_cast<const uint32_t(&)[8]>(lw[0]));
    st_global_v8(lp + 16, reinterpret_cast<const uint32_t(&)[8]>(lw[8]));
  } else {
    uint32_t hw[32], lw[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float h, l;
      split_tf32(a[j], h, l);
      hw[j] = __float_as_uint(h);
      lw[j] = __float_as_uint(l);
    }
    float* hp = reinterpret_cast<float*>(g.out) + poff;
    float* lp = reinterpret_cast<float*>(g.out_lo) + poff;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      st_global_v8(hp + 8 * q, reinterpret_cast<const uint32_t(&)[8]>(hw[8 * q]));
      st_global_v8(lp + 8 * q, reinterpret_cast<const uint32_t(&)[8]>(lw[8 * q]));
    }
  }
}

// The same slice through shared memory and TMA (fp16 planes).  With the 256-bit stores above every lane of a store
// instruction touches a different 128 B line, which the LSU data pipe serialises into 16 B wavefronts: 4096 of them
// per 128x128 tile, 75 % of the pipe's cycles on the short-K layer waves (ncu l1tex__data_pipe_lsu_wavefronts,
// profiles/r2t_epilogue_store_path.txt) and the reason the epilogue warps sat on the store scoreboard while the
// next tile's accumulators waited.  Here a lane writes its row's 64 B of one plane into the warp's 2 KB staging
// slab (16 B chunks XOR-swizzled the way CU_TENSOR_MAP_SWIZZLE_64B expects: chunk ^= (row >> 1) & 3, conflict-free)
// and one lane hands the [32 rows][32 columns] box to the TMA unit; the lo' plane follows through the same slab once
// the hi store has read it.  Rows past M are clipped by the tensor map.
// Two phases so that the caller can put independent work (sign bits, column sums) between the hi store's issue and the
// wait for it to have read the slab: phase 1 returns the packed lo' words.
__device__ __forceinline__ void store_slice_tma_hi(const CUtensorMap* o_hi, uint32_t slab, const float* a, int lane, int mrow0,
                                                   int cbase, uint32_t (&lw)[16]) {
  uint32_t w[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const __half2 h2 = __floats2half2_rn(a[2 * q], a[2 * q + 1]);
    const float2 hf = __half22float2(h2);
    const __half2 l2 = __floats2half2_rn((a[2 * q] - hf.x) * 2048.0f, (a[2 * q + 1] - hf.y) * 2048.0f);
    w[q] = *reinterpret_cast<const uint32_t*>(&h2);
    lw[q] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  const uint32_t row = slab + (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
  // (the caller made sure the slab is free: bulk_wait_read0 + __syncwarp before the slice)
#pragma unroll
  for (uint32_t j = 0; j < 4; ++j) sts_v4(row + ((j ^ sw) << 4), w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
  fence_async_smem();
  __syncwarp();
  if (lane == 0) {
    tma_store_3d(o_hi, slab, cbase & 63, mrow0, cbase >> 6);
    bulk_commit();
  }
}
__device__ __forceinline__ void store_slice_tma_lo(const CUtensorMap* o_lo, uint32_t slab, const uint32_t (&lw)[16], int lane,
                                                   int mrow0, int cbase) {
  const uint32_t row = slab + (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
  if (lane == 0) bulk_wait_read0();
  __syncwarp();
#pragma unroll
  for (uint32_t j = 0; j < 4; ++j) sts_v4(row + ((j ^ sw) << 4), lw[4 * j], lw[4 * j + 1], lw[4 * j + 2], lw[4 * j + 3]);
  fence_async_smem();
  __syncwarp();
  if (lane == 0) {
    tma_store_3d(o_lo, slab, cbase & 63, mrow0, cbase >> 6);
    bulk_commit();
  }
}

// Forward epilogue with planes out, WITHOUT a register transpose: lane = row keeps its 32 accumulators (bias already
// added by the caller), applies ReLU / dropout, forms the sign-bit word, splits pairs of values with packed conversions
// and hands its 32 columns of each plane to the slab + TMA store path (fp16) or writes them with 256-bit stores (TF32:
// 128 B per plane = 4 stores).  ~10 instructions per element against ~29 of the staged path (ncu: the short-K layer
// waves were issue-bound at 61 % issue utilisation writing 2.2 TB/s, profiles/r2e_gemm_waves_ncu_full.txt).
template <int FMT>
__device__ __forceinline__ void emit_slice_fwd_planes(const GemmParams& g, float* a, int lane, int mrow0, int cbase,
                                                      const CUtensorMap* o_hi, const CUtensorMap* o_lo, uint32_t slab) {
  const int my_row = mrow0 + lane;
  const int kbo = cbase >> 5;
  if (kbo >= g.out_nb32) return;                         // warp-uniform
  const uint32_t cmask = (cbase + 32 <= g.N) ? 0xffffffffu : ((cbase < g.N) ? ((1u << (g.N - cbase)) - 1u) : 0u);
  if (g.act == ADN_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j], 0.f);
  }
  if (g.drop_thresh != 0u) {
    // tf.layers.dropout in TRAIN mode (simple_dnn.py:80-81): x * 1/(1-rate) * keep; the mask is the counter-based hash
    // the oracle restates (oracle/adanet_oracle.py dropout_keep_mask): element index = row * out + col
    const uint32_t key = g.drop_key0 + (uint32_t)(*g.drop_step) * 0xC2B2AE3Du;
    const uint32_t base = (uint32_t)my_row * (uint32_t)g.N + (uint32_t)cbase;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      uint32_t x = (base + (uint32_t)j) ^ key;
      x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
      a[j] = (x >= g.drop_thresh) ? a[j] * g.drop_scale : 0.f;
    }
  }
  if (cmask != 0xffffffffu) {       // K padding of the next GEMM must be exact zeros
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (!((cmask >> j) & 1u)) a[j] = 0.f;
  }
  const bool tma = FMT == FMT_F16 && g.out_tma;
  uint32_t lw[16];
  if (tma) store_slice_tma_hi(o_hi, slab, a, lane, mrow0, cbase, lw);
  uint32_t bits = 0u;               // (the sign bits are formed while the TMA unit reads the hi slab)
#pragma unroll
  for (int j = 0; j < 32; ++j) bits |= (a[j] > 0.f) ? (1u << j) : 0u;
  if (my_row < g.M) g.out_bits[(size_t)kbo * g.M + my_row] = bits;
  if (tma) store_slice_tma_lo(o_lo, slab, lw, lane, mrow0, cbase);
  else if (my_row < g.M) store_row32_planes<FMT>(g, a, my_row, cbase);
}

// dX epilogue with planes out, without a register transpose: sign-bit ReLU mask, plane stores as in the forward
// epilogue (slab + TMA, or 256-bit stores from the row-owning lane), and the per-32-row column sums (the bias
// gradient of the layer below) by a butterfly over the warp: at distance w a lane keeps the half of its columns selected by bit w of its lane id and receives the partner's
// partial sums for them, so after five rounds lane l holds the sum of column l over the 32 rows (31 shuffles and
// adds per lane, fixed order).
template <int FMT>
__device__ __forceinline__ void emit_slice_mask_planes(const GemmParams& g, float* a, uint32_t mwq, int lane, int mrow0, int cbase,
                                                       const CUtensorMap* o_hi, const CUtensorMap* o_lo, uint32_t slab) {
  const int my_row = mrow0 + lane;
  const int kbo = cbase >> 5;
  if (kbo >= g.out_nb32) return;                         // warp-uniform
  const uint32_t cmask = (cbase + 32 <= g.N) ? 0xffffffffu : ((cbase < g.N) ? ((1u << (g.N - cbase)) - 1u) : 0u);
  const uint32_t keep = (my_row < g.M) ? (mwq & cmask) : 0u;     // rows past M contribute nothing to the column sums
  if (g.out_mul != 1.0f) {
#pragma unroll
    for (int j = 0; j < 32; ++j) a[j] *= g.out_mul;
  }
  if (keep != 0xffffffffu) {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (!((keep >> j) & 1u)) a[j] = 0.f;
  }
  const bool tma = FMT == FMT_F16 && g.out_tma;
  uint32_t lw[16];
  if (tma) store_slice_tma_hi(o_hi, slab, a, lane, mrow0, cbase, lw);
  else if (my_row < g.M) store_row32_planes<FMT>(g, a, my_row, cbase);
  if (g.colsum_part) {
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
      const bool upper = (lane & w) != 0;
#pragma unroll
      for (int j = 0; j < w; ++j) {
        const float mine = upper ? a[j + w] : a[j];
        const float send = upper ? a[j] : a[j + w];
        a[j] = mine + __shfl_xor_sync(0xffffffffu, send, w);
      }
    }
    const int col = cbase + lane;
    if (col < g.colsum_ld) g.colsum_part[(size_t)(mrow0 >> 5) * g.colsum_ld + col] = a[0];
  }
  if (tma) store_slice_tma_lo(o_lo, slab, lw, lane, mrow0, cbase);     // (after the column sums: they cover the hi store's read)
}

template <int FMT, int EPI>
__device__ __forceinline__ void emit_slice(const GemmParams& g, const bool OUT_PLANES, float* a, uint32_t mwq, float* stage,
                                           int lane, int mrow0, int cbase, int rows_ok, float* dense, bool dense_vec,
                                           const bool bias_in_acc = false, const CUtensorMap* o_hi = nullptr,
                                           const CUtensorMap* o_lo = nullptr) {
  if (EPI == EPI_BIAS_ACT && OUT_PLANES && bias_in_acc) {
    emit_slice_fwd_planes<FMT>(g, a, lane, mrow0, cbase, o_hi, o_lo, smem_u32(stage));
    return;
  }
  if (EPI == EPI_MASK && OUT_PLANES && bias_in_acc) {
    emit_slice_mask_planes<FMT>(g, a, mwq, lane, mrow0, cbase, o_hi, o_lo, smem_u32(stage));
    return;
  }
  constexpr int SW = 16;                   // staged columns per pass (2 KB per warp, two passes)
  constexpr int CH = SW / 4;               // 16 B chunks per staged row
  constexpr int RPI = 32 / CH;             // rows covered by one transposed instruction (8)
  const int cc = lane % CH;                // 16 B chunk (4 columns) this lane owns after the transpose
  const int rsub = lane / CH;
  const int my_row = mrow0 + lane;
  const int kbo = cbase >> 5;              // 32-column block of the output
  const bool live = (OUT_PLANES ? (kbo < g.out_nb32) : (cbase < g.N)) && rows_ok > 0;   // warp-uniform
  // valid columns of this slice as a bit mask (warp-uniform); all ones for interior tiles
  const uint32_t cmask = (cbase + 32 <= g.N) ? 0xffffffffu : ((cbase < g.N) ? ((1u << (g.N - cbase)) - 1u) : 0u);
  if (EPI == EPI_BIAS_ACT) {
    if (g.bias && !bias_in_acc) {
      if (cmask == 0xffffffffu && (reinterpret_cast<uintptr_t>(g.bias) & 15) == 0) {
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const float4 bv = __ldg(reinterpret_cast<const float4*>(g.bias + cbase) + jj);   // warp-uniform address
          a[4 * jj + 0] += bv.x; a[4 * jj + 1] += bv.y;
          a[4 * jj + 2] += bv.z; a[4 * jj + 3] += bv.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if ((cmask >> j) & 1u) a[j] += __ldg(g.bias + cbase + j);
      }
    }
    if (g.act == ADN_ACT_RELU) {
#pragma unroll
      for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j], 0.f);
    }
    if (OUT_PLANES) {
      uint32_t bits = 0u;
#pragma unroll
      for (int j = 0; j < 32; ++j) bits |= (a[j] > 0.f) ? (1u << j) : 0u;
      bits &= cmask;
      if (live && my_row < g.M) g.out_bits[(size_t)kbo * g.M + my_row] = bits;
    }
    if (cmask != 0xffffffffu) {       // K padding of the next GEMM must be exact zeros
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (!((cmask >> j) & 1u)) a[j] = 0.f;
    }
  } else {
    if (g.out_mul != 1.0f) {
#pragma unroll
      for (int j = 0; j < 32; ++j) a[j] *= g.out_mul;
    }
    if (EPI == EPI_MASK) {
      const uint32_t keep = mwq & cmask;
      if (keep != 0xffffffffu) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (!((keep >> j) & 1u)) a[j] = 0.f;
      }
    }
  }
  // chunk swizzle by row: both the row-wise float4 writes and the transposed float4 reads are bank-conflict free
#define ADN_SWZ(r) (((r) >> 1) & 3)
  float cs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int h = 0; h < 32 / SW; ++h) {
    {
      float4* srow = reinterpret_cast<float4*>(stage + lane * SW);
#pragma unroll
      for (int jj = 0; jj < CH; ++jj)
        srow[jj ^ ADN_SWZ(lane)] = make_float4(a[h * SW + 4 * jj], a[h * SW + 4 * jj + 1], a[h * SW + 4 * jj + 2],
                                               a[h * SW + 4 * jj + 3]);
    }
    __syncwarp();
    if (live) {
      const int c4 = h * SW + cc * 4;       // column offset inside the 32-column slice
      const int col = cbase + c4;
      cs[0] = cs[1] = cs[2] = cs[3] = 0.f;
      // plane element offset of (row mrow0 + rsub, column col): k-block-major, BK columns per k-block row
      constexpr int BK = Fmt<FMT>::BK;
      const size_t poff = OUT_PLANES ? ((size_t)(col / BK) * g.M + mrow0 + rsub) * BK + (col % BK) : 0;
#pragma unroll
      for (int i = 0; i < 32 / RPI; ++i) {
        const int r = rsub + RPI * i;
        const bool rv = (rows_ok == 32) || (r < rows_ok);
        float4 t = reinterpret_cast<const float4*>(stage + r * SW)[cc ^ ADN_SWZ(r)];
        float v[4] = {t.x, t.y, t.z, t.w};
        if (EPI == EPI_MASK) {
#pragma unroll
          for (int k = 0; k < 4; ++k) cs[k] += rv ? v[k] : 0.f;
        }
        if (rv) {
          if (OUT_PLANES) {
            if (FMT == FMT_F16) {
              __half hh[4], ll[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) split_f16(v[k], hh[k], ll[k]);
              __half* hp = reinterpret_cast<__half*>(g.out) + poff + (size_t)i * RPI * BK;
              __half* lp = reinterpret_cast<__half*>(g.out_lo) + poff + (size_t)i * RPI * BK;
              *reinterpret_cast<uint2*>(hp) = make_uint2(pack_h2(hh[0], hh[1]), pack_h2(hh[2], hh[3]));
              *reinterpret_cast<uint2*>(lp) = make_uint2(pack_h2(ll[0], ll[1]), pack_h2(ll[2], ll[3]));
            } else {
              float hh[4], ll[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) split_tf32(v[k], hh[k], ll[k]);
              float* hp = reinterpret_cast<float*>(g.out) + poff + (size_t)i * RPI * BK;
              float* lp = reinterpret_cast<float*>(g.out_lo) + poff + (size_t)i * RPI * BK;
              *reinterpret_cast<float4*>(hp) = make_float4(hh[0], hh[1], hh[2], hh[3]);
              *reinterpret_cast<float4*>(lp) = make_float4(ll[0], ll[1], ll[2], ll[3]);
            }
          } else {
            float* op = dense + (size_t)(mrow0 + r) * g.ldc + col;
            if (dense_vec && col + 3 < g.N) {
              *reinterpret_cast<float4*>(op) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (col + k < g.N) op[k] = v[k];
            }
          }
        }
      }
      if (EPI == EPI_MASK && g.colsum_part) {
        // rows of this lane: rsub + RPI*i; fold the lanes that own the same columns in a fixed order
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          cs[k] += __shfl_xor_sync(0xffffffffu, cs[k], 4);
          cs[k] += __shfl_xor_sync(0xffffffffu, cs[k], 8);
          cs[k] += __shfl_xor_sync(0xffffffffu, cs[k], 16);
        }
        if (rsub == 0) {
          float* cp = g.colsum_part + (size_t)(mrow0 >> 5) * g.colsum_ld + col;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (col + k < g.colsum_ld) cp[k] = cs[k];
        }
      }
    }
    __syncwarp();
  }
#undef ADN_SWZ
}

// ---------------------------------------------------------------------------------
// GEMM kernel (grouped): one persistent launch runs the tiles of up to MAX_GROUP independent GEMMs of
// the same epilogue kind -- the same layer of every candidate subnetwork of an AdaNet iteration -- so the
// launch, prologue and pipeline fill/drain are paid once per layer wave instead of once per candidate,
// and the short-K tiles of narrow candidates hide behind the long-K tiles of wide ones.
// Work items are numbered problem after problem; CTA c takes items c, c + grid, ... (every CTA gets the
// same share of every problem).  A group of one is the plain single-GEMM call.
// ---------------------------------------------------------------------------------
static constexpr int MAX_GROUP = 8;

struct alignas(64) Problem {
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
  CUtensorMap o_hi, o_lo;   // output planes as [32 rows][32 columns] store boxes (GemmParams::out_tma)
  GemmParams g;
  int item0;             // first work item of this problem
  int pad_[3];
};
struct alignas(64) Group {
  Problem p[MAX_GROUP];
  int n;                 // problems
  int total_items;
};

// advance `cur` to the problem that owns `item` (items are visited in increasing order).  `next0` caches the first item
// of the following problem in a register: the common case is one compare, not an indexed load from the parameter bank.
__device__ __forceinline__ int find_problem(const Group& grp, int cur, int item, int& next0) {
  while (item >= next0) {
    ++cur;
    next0 = (cur + 1 < grp.n) ? grp.p[cur + 1].item0 : 0x7fffffff;
  }
  return cur;
}
__device__ __forceinline__ int first_next0(const Group& grp) { return grp.n > 1 ? grp.p[1].item0 : 0x7fffffff; }

template <int FMT, int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
pl_gemm_kernel(const __grid_constant__ Group grp) {
  constexpr int BK = Fmt<FMT>::BK;
  constexpr int CHUNK = Fmt<FMT>::CHUNK;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem) & 1023u) != 0u) __trap();   // SWIZZLE_128B tiles must sit on 1024 B boundaries
  float* epi_stage = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + EPI_BYTES);
  uint64_t* full_bar = bars;                       // [STAGES]  TMA -> MMA
  uint64_t* empty_bar = bars + STAGES;             // [STAGES]  MMA -> TMA
  uint64_t* acc_full = bars + 2 * STAGES;          // [2]       MMA -> epilogue (chunk ready)
  uint64_t* acc_empty = bars + 2 * STAGES + 2;     // [2]       epilogue -> MMA (chunk drained), count EPI_WARPS
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int n_items = grp.total_items;

  if (warp == 0 && lane < grp.n) {       // every problem's descriptors: each CTA visits every problem
    tma_prefetch_desc(&grp.p[lane].a_hi);
    tma_prefetch_desc(&grp.p[lane].a_lo);
    tma_prefetch_desc(&grp.p[lane].b_hi);
    tma_prefetch_desc(&grp.p[lane].b_lo);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(smem_u32(&full_bar[s]), 1);
        mbar_init(smem_u32(&empty_bar[s]), 1);
      }
      for (int b = 0; b < 2; ++b) {
        mbar_init(smem_u32(&acc_full[b]), 1);
        mbar_init(smem_u32(&acc_empty[b]), EPI_WARPS);
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      int cur = 0, next0 = first_next0(grp);
      const uint32_t smem0 = smem_u32(smem);
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        cur = find_problem(grp, cur, item, next0);
        const Problem& pr = grp.p[cur];
        const GemmParams& g = pr.g;
        const Item it = decode_item(g, item - pr.item0);
        for (int kb = 0; kb < it.nkb; ++kb) {
          mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1);
          const uint32_t fb = smem_u32(&full_bar[s]);
          mbar_expect_tx(fb, STAGE_BYTES);
          const uint32_t base = smem0 + s * STAGE_BYTES;
          const int kc = it.kb0 + kb;
          // K-major box {BK, 128 rows, 1 kb} at (0, row0, kc); MN-major box {BK, BK rows, 128/BK kb} at (0, kc*BK, mn0/BK)
          const int a1 = g.a_mn ? kc * BK : it.m0, a2 = g.a_mn ? (it.m0 / BK) : kc;
          const int b1 = g.b_mn ? kc * BK : it.n0, b2 = g.b_mn ? (it.n0 / BK) : kc;
          tma_load_3d(&pr.a_hi, fb, base + 0 * TILE_BYTES, 0, a1, a2);
          tma_load_3d(&pr.a_lo, fb, base + 1 * TILE_BYTES, 0, a1, a2);
          tma_load_3d(&pr.b_hi, fb, base + 2 * TILE_BYTES, 0, b1, b2);
          tma_load_3d(&pr.b_lo, fb, base + 3 * TILE_BYTES, 0, b1, b2);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    // The warp runs the loop converged (all lanes wait on the barriers); only the issue is under
    // elect.sync, so every operand is warp-uniform.  The issue loop keeps ring counters incremental and
    // builds descriptors from 32-bit halves.
    {
      const uint32_t smem0 = smem_u32(smem);
      uint32_t s = 0, ph = 0, gchunk = 0;
      int cur = 0, next0 = first_next0(grp);
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        cur = find_problem(grp, cur, item, next0);
        const GemmParams& g = grp.p[cur].g;
        const Item it = decode_item(g, item - grp.p[cur].item0);
        // B_hi and B_lo tiles are adjacent in the stage, so ONE N=256 MMA computes a_hi x [b_hi | b_lo] (hi*hi into
        // columns [0,128), hi*lo into [128,256) of the chunk buffer) and a second N=128 MMA adds a_lo x b_hi to the
        // cross-term half: 20 KiB of operand reads per K step instead of 24 (the 128x128 single-CTA tile is
        // bound by shared-memory traffic, not by MMA issue), same 192 clk of tensor work.
        const uint32_t idesc256 = make_idesc<FMT>(BM, 2 * BN, g.a_mn, g.b_mn);
        const uint32_t idesc128 = make_idesc<FMT>(BM, BN, g.a_mn, g.b_mn);
        const uint32_t dah = desc_hi_word<FMT>(g.a_mn), dbh = desc_hi_word<FMT>(g.b_mn);
        const uint32_t a_lo0 = desc_lo_word<FMT>(smem0, g.a_mn);
        const uint32_t b_lo0 = desc_lo_word<FMT>(smem0 + 2 * TILE_BYTES, g.b_mn);
        const uint32_t a_step = g.a_mn ? Fmt<FMT>::MN_STEP : (32u >> 4);   // address-field advance per MMA
        const uint32_t b_step = g.b_mn ? Fmt<FMT>::MN_STEP : (32u >> 4);
        for (int kb = 0; kb < it.nkb; kb += CHUNK, ++gchunk) {
          const uint32_t b = gchunk & 1;
          mbar_wait(smem_u32(&acc_empty[b]), ((gchunk >> 1) & 1) ^ 1);      // chunk buffer drained
          tc_fence_after();
          const uint32_t acc = tmem_base + b * 256;     // [H: 128 cols | S: 128 cols]
          const int nk = min(CHUNK, it.nkb - kb);
          uint32_t accum = 0;                      // first MMA of the chunk overwrites both halves
          for (int kk = 0; kk < nk; ++kk) {
            mbar_wait(smem_u32(&full_bar[s]), ph);
            tc_fence_after();
            const uint32_t so = s * (STAGE_BYTES >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {          // 4 MMAs per 128 B k-block (K = 8 tf32 / 16 f16 each)
                const uint32_t a_hi = a_lo0 + so + k * a_step, a_lo = a_hi + (TILE_BYTES >> 4);
                const uint32_t b_hi = b_lo0 + so + k * b_step;
                umma<FMT>(acc, a_hi, b_hi, dah, dbh, idesc256, (k == 0) ? accum : 1u);       // hi*hi | hi*lo
                umma<FMT>(acc + 128, a_lo, b_hi, dah, dbh, idesc128, 1u);                    // + lo*hi
              }
              umma_commit(smem_u32(&empty_bar[s]));  // frees this smem stage when the MMAs retire
              if (kk == nk - 1) umma_commit(smem_u32(&acc_full[b]));   // chunk complete
            }
            __syncwarp();
            accum = 1u;
            if (++s == STAGES) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else {
    // ================= epilogue warps 2..17 =================
    const int quad = warp & 3;                       // TMEM lane quadrant a warp may read = warp % 4
    const int cgrp = (warp - 2) >> 2;                // which 32 of the tile's 128 columns
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const uint32_t col_base = (uint32_t)(cgrp * 32);
    float* stage = epi_stage + (warp - 2) * EPI_STAGE_FLOATS;
    uint32_t gchunk = 0;
    int cur = 0, next0 = first_next0(grp);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      cur = find_problem(grp, cur, item, next0);
      const GemmParams& g = grp.p[cur].g;
      const Item it = decode_item(g, item - grp.p[cur].item0);
      const int mrow0 = it.m0 + quad * 32;
      const int ncol0 = it.n0 + (int)col_base;        // first output column of this warp
      const int my_row = mrow0 + lane;
      // ReLU mask: one sign-bit word per (row, 32-column block), fetched before the accumulators are awaited
      uint32_t mw = 0xffffffffu;
      if (EPI == EPI_MASK && g.mask_bits) {
        const int kbo = ncol0 >> 5;
        mw = (my_row < g.M && kbo < g.out_nb32) ? __ldg(g.mask_bits + (size_t)kbo * g.M + my_row) : 0u;
      }
      float acc[32];
      if (EPI == EPI_BIAS_ACT && g.bias) {
        // the bias starts the accumulation (fetched while the first chunk is still in flight): warp-uniform loads
        if (ncol0 + 32 <= g.N && (reinterpret_cast<uintptr_t>(g.bias) & 15) == 0) {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            const float4 bv = __ldg(reinterpret_cast<const float4*>(g.bias + ncol0) + jj);
            acc[4 * jj + 0] = bv.x; acc[4 * jj + 1] = bv.y;
            acc[4 * jj + 2] = bv.z; acc[4 * jj + 3] = bv.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[j] = (ncol0 + j < g.N) ? __ldg(g.bias + ncol0 + j) : 0.f;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = 0.f;
      }
      const int nchunks = (it.nkb + CHUNK - 1) / CHUNK;
      for (int c = 0; c < nchunks; ++c, ++gchunk) {
        const uint32_t b = gchunk & 1;
        mbar_wait(smem_u32(&acc_full[b]), (gchunk >> 1) & 1);
        tc_fence_after();
        {
          uint32_t r0[32], r1[32];
          tmem_ld32_nowait(tmem_base + lane_base + b * 256 + col_base, r0);          // hi*hi partial sums of this chunk
          tmem_ld32_nowait(tmem_base + lane_base + b * 256 + 128 + col_base, r1);    // cross terms of this chunk
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r0[j]);   // fp32 RN adds
          if (FMT == FMT_F16) {
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] = fmaf(__uint_as_float(r1[j]), 1.0f / 2048.0f, acc[j]);   // lo' carries 2^11
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(r1[j]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&acc_empty[b]));
      }
      // ---- tile output: this warp's 32 rows x 32 columns ----
      float* dense = reinterpret_cast<float*>(g.out);
      if (EPI == EPI_PARTIAL) dense += (size_t)it.split * g.M * g.N;
      const bool out_planes = g.out_planes != 0;
      const bool dense_vec = !out_planes && ((g.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(dense) & 15) == 0);
      const int rows_ok = min(32, g.M - mrow0);          // warp-uniform; <= 0: nothing to write
      if (FMT == FMT_F16) {     // the previous slice's TMA store must have read the staging slab
        if (lane == 0) bulk_wait_read0();
        __syncwarp();
      }
      emit_slice<FMT, EPI>(g, out_planes, acc, mw, stage, lane, mrow0, ncol0, rows_ok, dense, dense_vec, true,
                           &grp.p[cur].o_hi, &grp.p[cur].o_lo);
    }
    if (FMT == FMT_F16 && lane == 0) bulk_wait0();    // stores complete before the CTA (and its shared memory) goes away
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------
// dense <-> planes conversion (inputs x / labels-side gradients / weights; everything
// between two GEMMs is written as planes by the producing epilogue instead)
// ---------------------------------------------------------------------------------
// src[rows, cols] row-major (times `scale`, a power of two) -> hi/lo[nkb][rows][BK] (zero padded in cols) +
// sign bits[nkb * BK/32][rows]
template <int FMT>
__global__ void __launch_bounds__(256)
split_kernel(const float* __restrict__ src, void* __restrict__ hi_, void* __restrict__ lo_, uint32_t* __restrict__ bits,
             int rows, int cols, int nkb, float scale, unsigned int* ovf) {
  constexpr int BK = Fmt<FMT>::BK;
  const int vec_per_row = nkb * (BK / 4);                // float4 per padded row; 8 consecutive threads = one sign word
  const int64_t nvec = (int64_t)rows * vec_per_row;
  const int64_t nvec_pad = (nvec + 31) & ~(int64_t)31;   // whole warps run the loop (shuffles below)
  const bool vec_src = ((cols & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  bool over = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec_pad; i += (int64_t)gridDim.x * blockDim.x) {
    const bool live = i < nvec;
    const int r = live ? (int)(i / vec_per_row) : 0;
    const int c = live ? (int)(i % vec_per_row) * 4 : 0;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (live) {
      if (vec_src && c + 3 < cols) {
        float4 t = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * cols + c));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] = (c + q < cols) ? __ldg(src + (size_t)r * cols + c + q) : 0.f;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] *= scale;
    }
    uint32_t nib = 0u;
#pragma unroll
    for (int q = 0; q < 4; ++q) nib |= (v[q] > 0.f) ? (1u << q) : 0u;
    uint32_t w = nib << (4 * (threadIdx.x & 7));
    w |= __shfl_xor_sync(0xffffffffu, w, 1);
    w |= __shfl_xor_sync(0xffffffffu, w, 2);
    w |= __shfl_xor_sync(0xffffffffu, w, 4);
    if (live) {
      const size_t dst = ((size_t)(c / BK) * rows + r) * BK + (c % BK);
      if (FMT == FMT_F16) {
        __half h[4], l[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          split_f16(v[q], h[q], l[q]);
          over |= f16_overflows(v[q]);
        }
        *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(hi_) + dst) = make_uint2(pack_h2(h[0], h[1]), pack_h2(h[2], h[3]));
        *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(lo_) + dst) = make_uint2(pack_h2(l[0], l[1]), pack_h2(l[2], l[3]));
      } else {
        float h[4], l[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) split_tf32(v[q], h[q], l[q]);
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(hi_) + dst) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(lo_) + dst) = make_float4(l[0], l[1], l[2], l[3]);
      }
      if ((threadIdx.x & 7) == 0) bits[(size_t)(c >> 5) * rows + r] = w;
    }
  }
  if (over) raise_overflow(ovf);
}

// hi/lo[nkb][rows][BK] -> dst[rows, cols] = hi + lo (tf32) | hi + 2^-11 lo' (f16)
template <int FMT>
__global__ void __launch_bounds__(256)
merge_kernel(const void* __restrict__ hi_, const void* __restrict__ lo_, float* __restrict__ dst, int rows, int cols, int nkb) {
  constexpr int BK = Fmt<FMT>::BK;
  const int64_t n = (int64_t)rows * nkb * BK;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int cb = (int)(i % BK);
    const int64_t t = i / BK;
    const int r = (int)(t % rows);
    const int c = (int)(t / rows) * BK + cb;
    if (c < cols) {
      if (FMT == FMT_F16)
        dst[(size_t)r * cols + c] = merge_f16(reinterpret_cast<const __half*>(hi_)[i], reinterpret_cast<const __half*>(lo_)[i]);
      else
        dst[(size_t)r * cols + c] = reinterpret_cast<const float*>(hi_)[i] + reinterpret_cast<const float*>(lo_)[i];
    }
  }
}

// ---------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------
__device__ unsigned int g_plane_overflow = 0u;

static PFN_cuTensorMapEncodeTiled g_encode = nullptr;
static unsigned int* g_ovf_addr = nullptr;
static std::atomic<int> g_format{-1};

int format() {
  int f = g_format.load();
  if (f >= 0) return f;
  const char* e = getenv("ADN_PLANES");
  f = (e && (!strcmp(e, "tf32") || !strcmp(e, "TF32"))) ? FMT_TF32 : FMT_F16;
  g_format.store(f);
  return f;
}
int set_format(int fmt) {
  if (fmt != FMT_TF32 && fmt != FMT_F16) return fail(ADN_ERR_INVALID, "adn_set_plane_format: bad format %d", fmt);
  g_format.store(fmt);
  return ADN_OK;
}
unsigned int* overflow_flag() { return g_ovf_addr; }

int read_overflow(int* out_host, int reset, cudaStream_t st) {
  if (!g_ovf_addr) return fail(ADN_ERR_CUDA, "pl: adn_init() was not called");
  unsigned int v = 0;
  ADN_CUDA(cudaMemcpyAsync(&v, g_ovf_addr, sizeof(v), cudaMemcpyDeviceToHost, st));
  if (reset) ADN_CUDA(cudaMemsetAsync(g_ovf_addr, 0, sizeof(v), st));
  ADN_CUDA(cudaStreamSynchronize(st));
  *out_host = (int)v;
  return ADN_OK;
}

int init() {
  static std::once_flag once;
  static int rc = ADN_OK;
  std::call_once(once, []() {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || fn == nullptr) {
      (void)cudaGetLastError();
      rc = fail(ADN_ERR_CUDA, "pl::init: cuTensorMapEncodeTiled entry point unavailable");
      return;
    }
    g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn);
    bool ok = true;
#define ADN_PL_ATTR(F, E) \
  ok = ok && (cudaFuncSetAttribute(pl_gemm_kernel<F, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) == cudaSuccess)
    ADN_PL_ATTR(FMT_TF32, EPI_BIAS_ACT); ADN_PL_ATTR(FMT_TF32, EPI_MASK); ADN_PL_ATTR(FMT_TF32, EPI_PARTIAL);
    ADN_PL_ATTR(FMT_F16, EPI_BIAS_ACT); ADN_PL_ATTR(FMT_F16, EPI_MASK); ADN_PL_ATTR(FMT_F16, EPI_PARTIAL);
#undef ADN_PL_ATTR
    if (!ok) {
      (void)cudaGetLastError();
      rc = fail(ADN_ERR_CUDA, "pl::init: cudaFuncSetAttribute(smem=%d) failed", SMEM_BYTES);
      return;
    }
    void* addr = nullptr;
    if (cudaGetSymbolAddress(&addr, g_plane_overflow) != cudaSuccess || !addr) {
      (void)cudaGetLastError();
      rc = fail(ADN_ERR_CUDA, "pl::init: cudaGetSymbolAddress(g_plane_overflow) failed");
      return;
    }
    g_ovf_addr = reinterpret_cast<unsigned int*>(addr);
  });
  return rc;
}

int64_t planes_bytes_fmt(int fmt, int64_t rows, int64_t cols) { return planes_bytes(fmt, rows, cols); }

// a plane tensor viewed as a GEMM operand
struct Operand {
  const void* hi;
  const void* lo;
  int64_t rows, nkb;
  int mn_major;
};
static Operand operand(int fmt, const void* planes, int64_t rows, int64_t cols, int mn_major) {
  const char* p = reinterpret_cast<const char*>(planes);
  return Operand{p, p + plane_bytes1(fmt, rows, cols), rows, ceil_div(cols, fmt_bk(fmt)), mn_major};
}

// ---- TMA descriptor cache (include/adanet_b200.h conventions): a descriptor depends only on (plane base, rows,
// k-blocks, majorness, format); the same few hundred recur on every eager step, eval pass and graph re-capture.
struct MapKey {
  const void* ptr;
  int64_t rows, nkb;
  int mn, fmt;
  bool operator==(const MapKey& o) const { return ptr == o.ptr && rows == o.rows && nkb == o.nkb && mn == o.mn && fmt == o.fmt; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<uintptr_t>(k.ptr) * 0x9E3779B97F4A7C15ull;
    h ^= (size_t)k.rows * 0xC2B2AE3D27D4EB4Full + ((size_t)k.nkb << 20) + ((size_t)k.mn << 1) + (size_t)k.fmt;
    return h ^ (h >> 29);
  }
};
static std::mutex g_map_mu;
static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;
static std::atomic<long long> g_map_hits{0}, g_map_misses{0};
long long map_cache_hits() { return g_map_hits.load(); }
long long map_cache_misses() { return g_map_misses.load(); }

static int make_map(int fmt, CUtensorMap* map, const void* plane, int64_t rows, int64_t nkb, int mn_major) {
  if (!g_encode) return fail(ADN_ERR_CUDA, "pl: adn_init() was not called");
  const MapKey key{plane, rows, nkb, mn_major, fmt};
  {
    std::lock_guard<std::mutex> lk(g_map_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) {
      *map = it->second;
      g_map_hits.fetch_add(1, std::memory_order_relaxed);
      return ADN_OK;
    }
  }
  const int bk = fmt_bk(fmt), es = fmt_esize(fmt);
  cuuint64_t gdim[3] = {(cuuint64_t)bk, (cuuint64_t)rows, (cuuint64_t)nkb};
  cuuint64_t gstride[2] = {(cuuint64_t)bk * es, (cuuint64_t)rows * bk * es};
  cuuint32_t box_k[3] = {(cuuint32_t)bk, 128u, 1u};
  cuuint32_t box_mn[3] = {(cuuint32_t)bk, (cuuint32_t)bk, (cuuint32_t)(128 / bk)};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  const CUtensorMapSwizzle sw = (mn_major && fmt == FMT_TF32) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = g_encode(map, fmt == FMT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                        const_cast<void*>(plane), gdim, gstride, mn_major ? box_mn : box_k, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ADN_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld nkb=%lld mn=%d fmt=%d", (int)r,
                                     (long long)rows, (long long)nkb, mn_major, fmt);
  g_map_misses.fetch_add(1, std::memory_order_relaxed);
  std::lock_guard<std::mutex> lk(g_map_mu);
  if (g_maps.size() > 16384) g_maps.clear();     // bounded: buffers come and go with plans
  g_maps.emplace(key, *map);
  return ADN_OK;
}

// output planes (fp16) as TMA store targets: [32 columns (64 B)][32 rows] boxes, SWIZZLE_64B in shared memory
static int make_store_map(CUtensorMap* map, const void* plane, int64_t rows, int64_t nkb) {
  if (!g_encode) return fail(ADN_ERR_CUDA, "pl: adn_init() was not called");
  const MapKey key{plane, rows, nkb, 2, FMT_F16};      // mn = 2: the store box
  {
    std::lock_guard<std::mutex> lk(g_map_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) {
      *map = it->second;
      g_map_hits.fetch_add(1, std::memory_order_relaxed);
      return ADN_OK;
    }
  }
  cuuint64_t gdim[3] = {64u, (cuuint64_t)rows, (cuuint64_t)nkb};
  cuuint64_t gstride[2] = {128u, (cuuint64_t)rows * 128u};
  cuuint32_t box[3] = {32u, 32u, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(plane), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ADN_ERR_CUDA, "cuTensorMapEncodeTiled (store box) failed (%d) rows=%lld nkb=%lld", (int)r,
                                     (long long)rows, (long long)nkb);
  g_map_misses.fetch_add(1, std::memory_order_relaxed);
  std::lock_guard<std::mutex> lk(g_map_mu);
  if (g_maps.size() > 16384) g_maps.clear();
  g_maps.emplace(key, *map);
  return ADN_OK;
}

// one GEMM of a group: operands + epilogue description (tiles / item numbering are filled at launch)
struct GemmDesc {
  Operand a, b;
  GemmParams g;
};

static int encode_maps(int fmt, const GemmDesc& d, CUtensorMap* a_hi, CUtensorMap* a_lo, CUtensorMap* b_hi, CUtensorMap* b_lo,
                       const char* what) {
  if ((reinterpret_cast<uintptr_t>(d.a.hi) | reinterpret_cast<uintptr_t>(d.a.lo) | reinterpret_cast<uintptr_t>(d.b.hi) |
       reinterpret_cast<uintptr_t>(d.b.lo)) & 127)
    return fail(ADN_ERR_INVALID, "%s: plane buffers must be 256 B aligned", what);
  int rc;
  if ((rc = make_map(fmt, a_hi, d.a.hi, d.a.rows, d.a.nkb, d.a.mn_major))) return rc;
  if ((rc = make_map(fmt, a_lo, d.a.lo, d.a.rows, d.a.nkb, d.a.mn_major))) return rc;
  if ((rc = make_map(fmt, b_hi, d.b.hi, d.b.rows, d.b.nkb, d.b.mn_major))) return rc;
  if ((rc = make_map(fmt, b_lo, d.b.lo, d.b.rows, d.b.nkb, d.b.mn_major))) return rc;
  return ADN_OK;
}

template <int FMT, int EPI>
static void launch_kernel(const Group& grp, int grid, cudaStream_t st) {
  pl_gemm_kernel<FMT, EPI><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(grp);
}

// n independent GEMMs of the same epilogue kind -> persistent launches of up to MAX_GROUP problems each
template <int EPI>
static int launch_group(int fmt, const GemmDesc* d, int n, cudaStream_t st, const char* what) {
  for (int i0 = 0; i0 < n; i0 += MAX_GROUP) {
    const int m = std::min(MAX_GROUP, n - i0);
    Group grp;
    memset(&grp, 0, sizeof(grp));
    int items = 0;
    for (int i = 0; i < m; ++i) {
      const GemmDesc& src = d[i0 + i];
      Problem& pr = grp.p[i];
      int rc = encode_maps(fmt, src, &pr.a_hi, &pr.a_lo, &pr.b_hi, &pr.b_lo, what);
      if (rc) return rc;
      pr.g = src.g;
      pr.g.out_tma = 0;
      if (fmt == FMT_F16 && EPI != EPI_PARTIAL && src.g.out_planes && (src.g.out_nb32 & 1) == 0 &&
          ((reinterpret_cast<uintptr_t>(src.g.out) | reinterpret_cast<uintptr_t>(src.g.out_lo)) & 127) == 0) {
        if ((rc = make_store_map(&pr.o_hi, src.g.out, src.g.M, src.g.out_nb32 / 2))) return rc;
        if ((rc = make_store_map(&pr.o_lo, src.g.out_lo, src.g.M, src.g.out_nb32 / 2))) return rc;
        pr.g.out_tma = 1;
      }
      pr.g.a_mn = src.a.mn_major;
      pr.g.b_mn = src.b.mn_major;
      pr.g.tiles_m = (int)ceil_div(pr.g.M, BM);
      pr.g.tiles_n = (int)ceil_div(pr.g.N, BN);
      pr.g.tiles = pr.g.tiles_m * pr.g.tiles_n;
      if ((int64_t)pr.g.tiles * pr.g.splits >= (1 << 21))
        return fail(ADN_ERR_UNSUPPORTED, "%s: %d work items exceed the decode range", what, pr.g.tiles * pr.g.splits);
      pr.g.inv_tiles = 1.0f / (float)pr.g.tiles;
      pr.g.inv_tiles_n = 1.0f / (float)pr.g.tiles_n;
      pr.g.ovf = g_ovf_addr;
      pr.item0 = items;
      items += pr.g.tiles_m * pr.g.tiles_n * pr.g.splits;
    }
    grp.n = m;
    grp.total_items = items;
    const int grid = std::min(items, sm_count());
    if (fmt == FMT_F16) launch_kernel<FMT_F16, EPI>(grp, grid, st);
    else launch_kernel<FMT_TF32, EPI>(grp, grid, st);
    ADN_CHECK_LAUNCH(what);
  }
  return ADN_OK;
}

int split(int fmt, const float* src, int64_t rows, int64_t cols, void* planes, int log2_scale, cudaStream_t st) {
  const int bk = fmt_bk(fmt);
  const int64_t nkb = ceil_div(cols, bk);
  const int64_t nvec = rows * nkb * (bk / 4);
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(nvec, 256), (int64_t)sm_count() * 16));
  const PlaneView v = plane_view(fmt, planes, rows, cols);
  const float scale = ldexpf(1.0f, log2_scale);
  if (fmt == FMT_F16)
    split_kernel<FMT_F16><<<blocks, 256, 0, st>>>(src, v.hi, v.lo, v.bits, (int)rows, (int)cols, (int)nkb, scale, g_ovf_addr);
  else
    split_kernel<FMT_TF32><<<blocks, 256, 0, st>>>(src, v.hi, v.lo, v.bits, (int)rows, (int)cols, (int)nkb, scale, g_ovf_addr);
  ADN_CHECK_LAUNCH("planes split");
  return ADN_OK;
}

int merge(int fmt, const void* planes, int64_t rows, int64_t cols, float* dst, cudaStream_t st) {
  const int bk = fmt_bk(fmt);
  const int64_t nkb = ceil_div(cols, bk);
  const int64_t n = rows * nkb * bk;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n, 256), (int64_t)sm_count() * 16));
  const PlaneView v = plane_view(fmt, const_cast<void*>(planes), rows, cols);
  if (fmt == FMT_F16) merge_kernel<FMT_F16><<<blocks, 256, 0, st>>>(v.hi, v.lo, dst, (int)rows, (int)cols, (int)nkb);
  else merge_kernel<FMT_TF32><<<blocks, 256, 0, st>>>(v.hi, v.lo, dst, (int)rows, (int)cols, (int)nkb);
  ADN_CHECK_LAUNCH("planes merge");
  return ADN_OK;
}

// dW split-K: the partial buffer bounds the split count (<= 16M floats, <= 64 splits)
static int max_dw_splits(int64_t in, int64_t out) {
  int64_t s = (16LL << 20) / std::max<int64_t>(1, in * out);
  if (s > MAX_SPLITS) s = MAX_SPLITS;
  if (s < 1) s = 1;
  return (int)s;
}

int64_t dense_bwd_workspace_bytes(int64_t batch, int64_t in, int64_t out) {
  int64_t b = align_up((int64_t)max_dw_splits(in, out) * in * out * (int64_t)sizeof(float), 256);   // dW split-K partials
  b += align_up(ceil_div(batch, 32) * in * (int64_t)sizeof(float), 256);                             // dx column sums per 32 rows
  b += align_up(64 * in * (int64_t)sizeof(float), 256);                                              // their second-level partials
  return b + 512;
}

int dense_fwd_group(int fmt, const FwdOp* ops, int n, int64_t batch, cudaStream_t st) {
  if (n <= 0) return ADN_OK;
  const int bk = fmt_bk(fmt);
  std::vector<GemmDesc> d((size_t)n);
  for (int i = 0; i < n; ++i) {
    const FwdOp& o = ops[i];
    GemmDesc& e = d[(size_t)i];
    e.a = operand(fmt, o.xp, batch, o.in, 0);       // A = x  [M=batch, K=in]  K-major
    e.b = operand(fmt, o.wp, o.in, o.out, 1);       // B = w  [K=in, N=out]    MN-major
    GemmParams g{};
    g.M = (int)batch; g.N = (int)o.out;
    g.total_kb = (int)ceil_div(o.in, bk); g.kb_per_split = g.total_kb; g.splits = 1;
    g.bias = o.bias; g.act = o.act;
    g.out_mul = 1.0f;
    if (o.dropout_rate > 0.f) {
      if (!o.yp || !o.dropout_step) return fail(ADN_ERR_INVALID, "pl dense_fwd: dropout needs planes out and a step counter");
      const double t = (double)o.dropout_rate * 4294967296.0;
      g.drop_thresh = t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
      if (g.drop_thresh == 0u) g.drop_thresh = 1u;
      g.drop_key0 = o.dropout_seed * 0x9E3779B1u + (uint32_t)o.dropout_layer * 0x85EBCA77u + 0x27D4EB2Fu;
      g.drop_scale = 1.0f / (1.0f - o.dropout_rate);
      g.drop_step = o.dropout_step;
    }
    if (o.yp) {
      const PlaneView v = plane_view(fmt, o.yp, batch, o.out);
      g.out_planes = 1;
      g.out = v.hi; g.out_lo = v.lo; g.out_nb32 = (int)bits_blocks(fmt, o.out);
      g.out_bits = v.bits;
    } else {
      g.out = o.y; g.ldc = (int)o.out;
    }
    e.g = g;
  }
  return launch_group<EPI_BIAS_ACT>(fmt, d.data(), n, st, "pl dense_fwd gemm");
}

int dense_bwd_group(int fmt, const BwdOp* ops, int n, int64_t batch, cudaStream_t st) {
  if (n <= 0) return ADN_OK;
  const int bk = fmt_bk(fmt);
  const int workers = sm_count();
  struct Carve { float* part; float* cspart; float* cspart2; int splits; };
  std::vector<Carve> cv((size_t)n);
  std::vector<GemmDesc> dwd, dxd;
  // Split-K over the batch for the dW GEMMs of the group.  Work items of one launch are dealt round-robin to the
  // CTAs (item j -> CTA j % grid), so the launch takes as long as its most loaded CTA.  Every problem uses the
  // k-blocks-per-item `kps` (raised to its own partial-buffer bound), and kps is chosen by evaluating, for every
  // candidate split count, the exact round-robin load (k-blocks + a per-item pipeline fill/drain + epilogue
  // allowance) plus the cost of the fixed-order reduction of the partial sums (bytes at ~2.5 TB/s; one k-block
  // of MMA work is ~0.4 us).  (A k-block is 4 MMA steps in either format.)
  const int64_t kb_b = ceil_div(batch, bk);
  int64_t best_kps = kb_b;
  {
    static std::mutex mu;
    static std::unordered_map<std::string, int64_t> memo;      // the same waves recur every step / capture
    std::string key = std::to_string(batch) + ":" + std::to_string(fmt);
    for (int i = 0; i < n; ++i)
      if (ops[i].dw) key += "," + std::to_string(ops[i].in) + "x" + std::to_string(ops[i].out);
    bool hit = false;
    {
      std::lock_guard<std::mutex> lk(mu);
      auto it = memo.find(key);
      if (it != memo.end()) { best_kps = it->second; hit = true; }
    }
    if (!hit) {
      const double kItemOverhead = 6.0;          // k-block equivalents per work item
      const double kReduceKbPerByte = 1.0 / (2.5e6 * 0.4);     // k-block equivalents per byte of partials read
      double best_t = 1e30;
      std::vector<double> load((size_t)workers);
      int64_t last_kps = -1;
      for (int s0 = 1; s0 <= MAX_SPLITS && s0 <= kb_b; ++s0) {
        const int64_t kps = ceil_div(kb_b, s0);
        if (kps == last_kps) continue;
        last_kps = kps;
        std::fill(load.begin(), load.end(), 0.0);
        int64_t item = 0;
        double reduce_bytes = 0.0;
        bool any = false;
        for (int i = 0; i < n; ++i) {
          if (!ops[i].dw) continue;
          any = true;
          const int64_t k_i = std::max<int64_t>(kps, ceil_div(kb_b, max_dw_splits(ops[i].in, ops[i].out)));
          const int64_t s_i = ceil_div(kb_b, k_i);
          const int64_t tiles = ceil_div(ops[i].in, BM) * ceil_div(ops[i].out, BN);
          for (int64_t sp = 0; sp < s_i; ++sp) {
            const double kb_item = (double)(std::min(kb_b, (sp + 1) * k_i) - sp * k_i);
            for (int64_t t = 0; t < tiles; ++t, ++item) load[(size_t)(item % workers)] += kb_item + kItemOverhead;
          }
          if (s_i > 1) reduce_bytes += (double)(s_i + 1) * (double)ops[i].in * (double)ops[i].out * 4.0;
        }
        if (!any) break;
        const double t = *std::max_element(load.begin(), load.end()) + reduce_bytes * kReduceKbPerByte +
                         (reduce_bytes > 0 ? 10.0 : 0.0);
        if (t < best_t) { best_t = t; best_kps = kps; }
      }
      std::lock_guard<std::mutex> lk(mu);
      if (memo.size() > 4096) memo.clear();
      memo[key] = best_kps;
    }
  }
  for (int i = 0; i < n; ++i) {
    const BwdOp& o = ops[i];
    if (!o.ws || o.ws_bytes < dense_bwd_workspace_bytes(batch, o.in, o.out))
      return fail(ADN_ERR_WORKSPACE, "pl dense_bwd: op %d workspace %lld < %lld bytes", i, (long long)o.ws_bytes,
                  (long long)dense_bwd_workspace_bytes(batch, o.in, o.out));
    const float unscale = ldexpf(1.0f, -o.dz_log2_scale);
    char* p = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(o.ws) + 255) & ~(uintptr_t)255);
    const int max_s = max_dw_splits(o.in, o.out);
    Carve& c = cv[(size_t)i];
    c.part = reinterpret_cast<float*>(p);
    p += align_up((int64_t)max_s * o.in * o.out * (int64_t)sizeof(float), 256);
    c.cspart = reinterpret_cast<float*>(p);
    p += align_up(ceil_div(batch, 32) * o.in * (int64_t)sizeof(float), 256);
    c.cspart2 = reinterpret_cast<float*>(p);
    c.splits = 1;
    if (o.dw) {
      // ---- dW[in,out] = X^T dZ : A = Xp MN-major (M=in), B = dZp MN-major (N=out), K = batch, split-K ----
      GemmDesc e;
      e.a = operand(fmt, o.xp, batch, o.in, 1);
      e.b = operand(fmt, o.dzp, batch, o.out, 1);
      GemmParams g{};
      g.M = (int)o.in; g.N = (int)o.out; g.ldc = (int)o.out;
      g.total_kb = (int)kb_b; g.kb_per_split = (int)std::max<int64_t>(best_kps, ceil_div(kb_b, max_s));
      g.splits = (int)ceil_div(kb_b, g.kb_per_split);
      g.out = (g.splits == 1) ? o.dw : c.part;
      g.out_mul = (g.splits == 1) ? unscale : 1.0f;      // partials are un-scaled by the fixed-order reduction
      c.splits = g.splits;
      e.g = g;
      dwd.push_back(e);
    }
    if (o.dxp || o.dx) {
      // ---- dX[batch,in] = dZ W^T : A = dZp K-major (K=out), B = Wp K-major (N=in, K=out); ReLU mask = sign bits of X ----
      GemmDesc e;
      e.a = operand(fmt, o.dzp, batch, o.out, 0);
      e.b = operand(fmt, o.wp, o.in, o.out, 0);
      GemmParams g{};
      g.M = (int)batch; g.N = (int)o.in;
      g.total_kb = (int)ceil_div(o.out, bk); g.kb_per_split = g.total_kb; g.splits = 1;
      g.mask_bits = o.x_relu_mask ? bits_of(fmt, o.xp, batch, o.in) : nullptr;
      g.out_nb32 = (int)bits_blocks(fmt, o.in);
      g.colsum_part = o.dx_colsum ? c.cspart : nullptr;
      g.colsum_ld = (int)o.in;
      if (o.dxp) {
        const PlaneView v = plane_view(fmt, o.dxp, batch, o.in);
        g.out_planes = 1;
        g.out = v.hi; g.out_lo = v.lo;
        g.out_mul = o.dx_mul;              // the gradient keeps its scale while it stays in plane format
      } else {
        g.out = o.dx; g.ldc = (int)o.in;
        g.out_mul = unscale * o.dx_mul;    // dense fp32 leaves the plane pipeline: true magnitude
      }
      e.g = g;
      dxd.push_back(e);
    }
  }
  int rc;
  if (!dwd.empty()) {
    if ((rc = launch_group<EPI_PARTIAL>(fmt, dwd.data(), (int)dwd.size(), st, "pl dW gemm"))) return rc;
    std::vector<simt::ReduceJob> jobs;
    for (int i = 0; i < n; ++i)
      if (ops[i].dw && cv[(size_t)i].splits > 1)
        jobs.push_back(simt::ReduceJob{cv[(size_t)i].part, ops[i].dw, ops[i].in * ops[i].out, cv[(size_t)i].splits,
                                       ops[i].in * ops[i].out, ldexpf(1.0f, -ops[i].dz_log2_scale)});
    if ((rc = simt::reduce_partials_group(jobs.data(), (int)jobs.size(), st))) return rc;
  }
  if (!dxd.empty()) {
    if ((rc = launch_group<EPI_MASK>(fmt, dxd.data(), (int)dxd.size(), st, "pl dX gemm"))) return rc;
    // column sums of each [ceil(batch/32), in] partial matrix, fixed order
    std::vector<simt::ColsumJob> jobs;
    for (int i = 0; i < n; ++i)
      if (ops[i].dx_colsum && (ops[i].dxp || ops[i].dx))
        jobs.push_back(simt::ColsumJob{cv[(size_t)i].cspart, ops[i].dx_colsum, ceil_div(batch, 32), ops[i].in,
                                       cv[(size_t)i].cspart2, ops[i].dxp ? ldexpf(1.0f, -ops[i].dz_log2_scale) : 1.0f});
    if ((rc = simt::colsum_group(jobs.data(), (int)jobs.size(), st))) return rc;
  }
  return ADN_OK;
}

int dense_fwd(int fmt, const void* xp, const void* wp, const float* bias, void* yp, float* y, int64_t batch, int64_t in,
              int64_t out, int act, cudaStream_t st) {
  FwdOp op{xp, wp, bias, yp, y, in, out, act};
  return dense_fwd_group(fmt, &op, 1, batch, st);
}

int dense_bwd(int fmt, const void* xp, const void* wp, const void* dzp, void* dxp, float* dx, float* dx_colsum, float* dw,
              int64_t batch, int64_t in, int64_t out, int x_relu_mask, int dz_log2_scale, void* ws, int64_t ws_bytes,
              cudaStream_t st) {
  BwdOp op{xp, wp, dzp, dxp, dx, dx_colsum, dw, in, out, x_relu_mask, dz_log2_scale, ws, ws_bytes};
  return dense_bwd_group(fmt, &op, 1, batch, st);
}

}  // namespace pl
}  // namespace adn
