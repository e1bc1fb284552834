// K6b: the SimpleCNN stem forward as a tcgen05 implicit GEMM (same contract as conv_stem_fwd_kernel in
// conv_stem.cu, which stays as the exact-fp32 cross-check path: ADN_CONV_PATH=simt).
//
// Formulation: rows = POOLED pixels, not conv positions.  For one pooled pixel the four conv positions of its 2x2
// window read a 4x4xCin input patch, so
//     acc[p][(pos, f)] = sum_k A[p][k] * W'[k][(pos, f)],   k = (i, j, c) over the 4x4xCin patch (K = 16*Cin),
//     W'[(i,j,c)][(dy,dx,f)] = w[i-dy][j-dx][c][f]  (zero outside the 3x3 support),   N = 4*F,
// is a [128 x K] x [K x N] GEMM per 128 pooled pixels whose accumulator row holds exactly what the epilogue thread
// of the SIMT kernel holds in registers: 4 positions x F filters of its own pooled pixel.  Bias, ReLU, the 2x2
// max, the arg-max, the TF32 hi/lo split and the plane stores therefore happen in one thread per pooled pixel,
// straight out of TMEM, with no cross-lane traffic.  The price is 1.78x the minimal MACs (zeros in W'), irrelevant
// at 3 x 6 tcgen05.mma (M128 N64 K8) per tile.
//
// fp32 accuracy: 3xTF32 (a_hi b_hi + a_lo b_hi + a_hi b_lo), K <= 48, one TMEM accumulator.
//
// Per CTA (512 threads = 4 warpgroups, 1 CTA per SM, images grid-strided): the image is staged zero-padded in shared
// memory with cp.async (a ring of 2 or 4 images).  Two builder warpgroups each take a tile of 128 pooled pixels: every
// thread gathers its own A row from the staged image (LDS.64), splits it and writes hi / lo in the canonical K-major
// SWIZZLE_128B layout (16-byte chunk index XOR row%8 -- what TMA would have produced), fence.proxy.async, one elected
// thread issues the MMAs and commits to the accumulator's mbarrier.  Two epilogue warpgroups read their accumulator
// rows with tcgen05.ld (warp w reads TMEM lanes 32(w%4)..) and run the epilogue while the builders fill the next
// tile.  W' (hi / lo, K-major) is built once per CTA.  The backward is the SIMT kernel in conv_stem.cu.
#include "common.cuh"
#include "plane_fmt.cuh"

namespace adn {
namespace convtc {

static constexpr int TILE_BYTES = 128 * 128;   // one k-block (32 floats) of a 128-row K-major SWIZZLE_128B tile

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float rna_tf32(float v) {
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
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
      else if (now - t0 > 4000000000LL) __trap();
    }
  }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void wg_barrier(int wg) { asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory"); }
// K-major SWIZZLE_128B smem descriptor (cute::UMMA::SmemDescriptor): start >> 4 | LBO(unused)=1 << 16 |
// SBO = 1024 B >> 4 at [32,46) | version 1 at [46,48) | layout type 2 at [61,64)
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint32_t desc_hi() { return (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29); }
// kind::tf32 instruction descriptor: D=f32, A=B=tf32, both K-major, N>>3 at [17,23), M>>4 at [24,29)
__device__ __forceinline__ uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint32_t da, uint32_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %4, p;\n\t}"
      ::"r"(tmem_d), "r"(da), "r"(db), "r"(desc_hi()), "r"(idesc), "r"(accum)
      : "memory");
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
// byte offset of element (row, k) inside one k-block tile ([rows][32 floats], SWIZZLE_128B)
__device__ __forceinline__ uint32_t sw128(int row, int k) {
  return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((((k >> 2) ^ (row & 7)) & 7) << 4) + ((k & 3) << 2));
}

template <int CIN>
__device__ __forceinline__ void stage_image(float* s_img, const float* img, int H, int W, int tid, int nthreads) {
  const int row = W * CIN;
  const int prow = (W + 2) * CIN;
  const int lane = tid & 31;
  for (int y = tid >> 5; y < H; y += nthreads / 32) {
    const float* src = img + y * row;
    float* dst = s_img + (y + 1) * prow + CIN;
    for (int r = lane; r < row; r += 32) cp_async4(dst + r, src + r);
  }
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&r)[8]) {
  uint32_t u[8];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) r[i] = __uint_as_float(u[i]);
}

static constexpr int FWD_THREADS = 512;
// staged-image ring depth of the forward: 4 where shared memory allows (F = 16), else 2
__host__ __device__ constexpr int fwd_image_buffers(int f) { return f == 16 ? 4 : 2; }

// Forward, warp specialised.  512 threads = 4 warpgroups over two pipeline slots s = 0, 1 (a slot = one A tile
// buffer + two TMEM accumulators):
//   warpgroup s     (builders of slot s): stage images (with the other builders), gather / split / swizzle the A
//                   rows of a tile, issue the MMAs of the tile (one elected thread) and commit to acc_full[s][a];
//   warpgroup 2 + s (epilogue of slot s): wait acc_full[s][a], tcgen05.ld the accumulator, release it (acc_free), then
//                   bias / ReLU / pool / split / store while the builders are already on the next tile.
// Shared memory (from a 1024-aligned base): W' hi|lo [2][KB][N][128 B]; A per slot hi|lo [2][KB][16 KB]; two padded
// images; bias; mbarriers acc_full[2][2], acc_free[2][2]; TMEM slot.
template <int CIN, int F>
__global__ void __launch_bounds__(FWD_THREADS, 1)
conv_stem_tc_fwd_kernel(const float* __restrict__ images, const float* __restrict__ kernel, const float* __restrict__ bias,
                        const pl::PlaneView pv, unsigned int* ovf,
                        uint32_t* __restrict__ argmax, int64_t B, int H, int W) {
  constexpr int K = 16 * CIN;              // 4x4xCIN patch
  constexpr int KB = (K + 31) / 32;        // k-blocks of 32 floats (128 B swizzle atoms)
  constexpr int N = 4 * F;                 // (pool position, filter)
  constexpr int NB = N * 128;              // bytes of one k-block of W'
  constexpr int TMEM_COLS = 4 * N < 32 ? 32 : 4 * N;   // 2 slots x 2 accumulators of N columns (N = 64 / 128 -> 256 / 512)
  constexpr int NBUF = fwd_image_buffers(F);           // ring of staged images: the fetch of image i+NBUF-1 runs under image i
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_w = base;                                  // [2 planes][KB][N][128 B]
  uint8_t* s_a = s_w + 2 * KB * NB;                     // [2 slots][2 planes][KB][16 KB]
  const int pimg = (H + 2) * (W + 2) * CIN;
  float* s_img0 = reinterpret_cast<float*>(s_a + 2 * 2 * KB * TILE_BYTES);
  float* s_b = s_img0 + NBUF * pimg;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_b + F);      // [0,4) acc_full[slot][acc], [4,8) acc_free[slot][acc]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_bar + 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wgi = tid >> 7, r = tid & 127;
  const int slot = wgi & 1;
  const bool builder = wgi < 2;
  // ---- once per CTA: W' (hi / lo, K-major swizzled), bias, zero borders of the image buffers, barriers, TMEM ----
  for (int idx = tid; idx < N * K; idx += FWD_THREADS) {
    const int n = idx / K, k = idx - n * K;
    const int pos = n / F, f = n - pos * F;
    const int c = k % CIN, ij = k / CIN;
    const int ky = (ij >> 2) - (pos >> 1), kx = (ij & 3) - (pos & 1);
    const float v = (ky >= 0 && ky < 3 && kx >= 0 && kx < 3) ? kernel[((ky * 3 + kx) * CIN + c) * F + f] : 0.f;
    const float h = rna_tf32(v);
    const uint32_t off = (uint32_t)(k >> 5) * NB + sw128(n, k & 31);
    *reinterpret_cast<float*>(s_w + off) = h;
    *reinterpret_cast<float*>(s_w + KB * NB + off) = rna_tf32(v - h);
  }
  for (int i = tid; i < F; i += FWD_THREADS) s_b[i] = bias[i];
  for (int i = tid; i < NBUF * pimg; i += FWD_THREADS) s_img0[i] = 0.f;
  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < 4; ++i) mbar_init(smem_u32(&s_bar[i]), 1);
      for (int i = 4; i < 8; ++i) mbar_init(smem_u32(&s_bar[i]), 128);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_async_smem();          // W' was written through the generic proxy, the MMAs read it through the async proxy
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // one full / free barrier pair PER ACCUMULATOR: a full barrier can then never run two phases ahead of the epilogue
  // (the next commit to the same accumulator needs the epilogue's release of the previous one)
  const uint32_t acc_full0 = smem_u32(&s_bar[2 * slot]);
  const uint32_t acc_free0 = smem_u32(&s_bar[4 + 2 * slot]);

  const int PH = H / 2, PW = W / 2, P = PH * PW;
  const int tiles = (P + 127) / 128;
  const int prow = (W + 2) * CIN;
  const int64_t img_elems = (int64_t)H * W * CIN;

  if (builder) {
    // =========================== builders: images -> A tiles -> MMAs ===========================
    const uint32_t idesc = make_idesc(128, N);
    const uint32_t w_addr = smem_u32(s_w);
    uint8_t* a_hi = s_a + slot * (2 * KB * TILE_BYTES);
    uint8_t* a_lo = a_hi + KB * TILE_BYTES;
    const uint32_t a_addr = smem_u32(a_hi);
    const int btid = tid;                      // 0..255 among the builders
    uint32_t n_tiles = 0;                      // tiles this slot has issued so far
    int64_t b = blockIdx.x;
    for (int i = 0; i < NBUF - 1; ++i) {       // prologue: the first NBUF-1 images of this CTA
      const int64_t bi = b + (int64_t)i * gridDim.x;
      if (bi < B) stage_image<CIN>(s_img0 + i * pimg, images + bi * img_elems, H, W, btid, 256);
      cp_async_commit();
    }
    int buf = 0;
    for (; b < B; b += gridDim.x, buf = (buf + 1 == NBUF) ? 0 : buf + 1) {
      cp_async_wait<NBUF - 2>();                       // this thread's copies of image b have landed
      asm volatile("bar.sync 3, 256;" ::: "memory");   // image b is visible to both builder warpgroups; image b-1 is no longer read
      const int64_t nb = b + (int64_t)(NBUF - 1) * gridDim.x;
      const int pbuf = (buf == 0) ? NBUF - 1 : buf - 1;    // the buffer image b-1 used
      if (nb < B) stage_image<CIN>(s_img0 + pbuf * pimg, images + nb * img_elems, H, W, btid, 256);
      cp_async_commit();
      const float* s_img = s_img0 + buf * pimg;
      for (int tile = slot; tile < tiles; tile += 2, ++n_tiles) {
        const int p = tile * 128 + r;
        const bool valid = p < P;
        const int py = valid ? p / PW : 0, px = valid ? p - py * PW : 0;
        const float* patch = s_img + (2 * py) * prow + (2 * px) * CIN;
        const uint32_t rowoff = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128);
        // the previous tile's MMAs must have finished reading this slot's A buffer
        if (n_tiles > 0) mbar_wait(acc_full0 + 8 * ((n_tiles - 1) & 1u), ((n_tiles - 1) >> 1) & 1u);
#pragma unroll
        for (int q = 0; q < K / 4; ++q) {
          const int i = (CIN == 3) ? q / 3 : q;
          const int o = (CIN == 3) ? (q % 3) * 4 : 0;
          const float2 v0 = *reinterpret_cast<const float2*>(patch + i * prow + o);        // 8-byte aligned (W even)
          const float2 v1 = *reinterpret_cast<const float2*>(patch + i * prow + o + 2);
          float4 h4, l4;
          h4.x = rna_tf32(v0.x); l4.x = rna_tf32(v0.x - h4.x);
          h4.y = rna_tf32(v0.y); l4.y = rna_tf32(v0.y - h4.y);
          h4.z = rna_tf32(v1.x); l4.z = rna_tf32(v1.x - h4.z);
          h4.w = rna_tf32(v1.y); l4.w = rna_tf32(v1.y - h4.w);
          const uint32_t off = (uint32_t)(q >> 3) * TILE_BYTES + rowoff + (uint32_t)((((q & 7) ^ (r & 7)) & 7) << 4);
          *reinterpret_cast<float4*>(a_hi + off) = h4;
          *reinterpret_cast<float4*>(a_lo + off) = l4;
        }
        fence_async_smem();
        wg_barrier(slot);
        if ((warp & 3) == 0) {
          if (elect_one()) {
            const uint32_t accsel = n_tiles & 1u;
            // the epilogue must have drained this accumulator (tile n_tiles - 2); a fresh barrier passes at parity 1
            mbar_wait(acc_free0 + 8 * accsel, ((n_tiles >> 1) & 1u) ^ 1u);
            tc_fence_after();
            const uint32_t tmem_acc = tmem_base + (uint32_t)((slot * 2 + accsel) * N);
            uint32_t accum = 0;
#pragma unroll
            for (int prod = 0; prod < 3; ++prod) {       // a_hi b_hi, a_lo b_hi, a_hi b_lo
              const uint32_t aa = a_addr + (prod == 1 ? KB * TILE_BYTES : 0);
              const uint32_t ww = w_addr + (prod == 2 ? KB * NB : 0);
#pragma unroll
              for (int ks = 0; ks < K / 8; ++ks) {
                const uint32_t da = desc_lo(aa + (ks >> 2) * TILE_BYTES + (ks & 3) * 32);
                const uint32_t db = desc_lo(ww + (ks >> 2) * NB + (ks & 3) * 32);
                umma_tf32(tmem_acc, da, db, idesc, accum);
                accum = 1;
              }
            }
            umma_commit(acc_full0 + 8 * accsel);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // =========================== epilogue: accumulator -> pooled planes ===========================
    const int64_t words_per_row = (int64_t)P * F / 16;
    uint32_t n_tiles = 0;
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
      for (int tile = slot; tile < tiles; tile += 2, ++n_tiles) {
        const int p = tile * 128 + r;
        const bool valid = p < P;
        const uint32_t accsel = n_tiles & 1u;
        const uint32_t tmem_row = tmem_base + (uint32_t)((slot * 2 + accsel) * N) + ((uint32_t)((warp & 3) * 32) << 16);
        mbar_wait(acc_full0 + 8 * accsel, (n_tiles >> 1) & 1u);
        tc_fence_after();
#pragma unroll 1
        for (int f0 = 0; f0 < F; f0 += 16) {
          uint32_t sign = 0u, arg = 0u;
          const int64_t col0 = (int64_t)p * F + f0;
#pragma unroll
          for (int f8 = 0; f8 < 16; f8 += 8) {
            float a0[8], a1[8], a2[8], a3[8];
            tmem_ld8(tmem_row + (uint32_t)(0 * F + f0 + f8), a0);
            tmem_ld8(tmem_row + (uint32_t)(1 * F + f0 + f8), a1);
            tmem_ld8(tmem_row + (uint32_t)(2 * F + f0 + f8), a2);
            tmem_ld8(tmem_row + (uint32_t)(3 * F + f0 + f8), a3);
            tmem_ld_wait();
            if (f0 + 16 >= F && f8 == 8) {       // last read of this accumulator: hand it back to the MMA issuer
              tc_fence_before();
              mbar_arrive(acc_free0 + 8 * accsel);
            }
            float outv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float bv = s_b[f0 + f8 + j];
              float m = a0[j] + bv;
              uint32_t a = 0u;
              const float m1 = a1[j] + bv, m2 = a2[j] + bv, m3 = a3[j] + bv;
              if (m1 > m) { m = m1; a = 1u; }
              if (m2 > m) { m = m2; a = 2u; }
              if (m3 > m) { m = m3; a = 3u; }
              m = fmaxf(m, 0.f);
              sign |= (m > 0.f) ? (1u << (f8 + j)) : 0u;
              arg |= a << (2 * (f8 + j));
              outv[j] = m;
            }
            if (valid) pl::plane_store8(pv, b, col0 + f8, outv, ovf);
          }
          if (valid) {
            reinterpret_cast<uint16_t*>(pv.bits)[((col0 >> 5) * B + b) * 2 + ((col0 >> 4) & 1)] = (uint16_t)sign;
            argmax[b * words_per_row + (col0 >> 4)] = arg;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

template <int CIN, int F>
static size_t smem_bytes(int h, int w) {
  constexpr int K = 16 * CIN, KB = (K + 31) / 32, N = 4 * F;
  return 1024 + (size_t)2 * KB * N * 128 + (size_t)2 * 2 * KB * TILE_BYTES +
         (size_t)fwd_image_buffers(F) * (h + 2) * (w + 2) * CIN * 4 + F * 4 + 8 * 8 + 16;
}

template <int CIN, int F>
static int launch(const float* images, const float* kernel, const float* bias, const pl::PlaneView pv,
                  uint32_t* argmax, int64_t batch, int h, int w, cudaStream_t st) {
  const size_t smem = smem_bytes<CIN, F>(h, w);
  auto kern = conv_stem_tc_fwd_kernel<CIN, F>;
  const int64_t cap = sm_count();
  const int grid = (int)(batch < cap ? batch : cap);
  kern<<<grid, FWD_THREADS, smem, st>>>(images, kernel, bias, pv, pl::overflow_flag(), argmax, batch, h, w);
  ADN_CHECK_LAUNCH("conv_stem_tc_fwd");
  return ADN_OK;
}

// raised once from adn_init (never inside a stream capture, see conv::init)
int init() {
#define ADN_CONVTC_ATTR(K) ADN_CUDA(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024))
  ADN_CONVTC_ATTR((conv_stem_tc_fwd_kernel<1, 16>)); ADN_CONVTC_ATTR((conv_stem_tc_fwd_kernel<3, 16>));
  ADN_CONVTC_ATTR((conv_stem_tc_fwd_kernel<1, 32>)); ADN_CONVTC_ATTR((conv_stem_tc_fwd_kernel<3, 32>));
#undef ADN_CONVTC_ATTR
  return ADN_OK;
}

// true when the tcgen05 path covers the shape (else the caller takes the SIMT kernel)
bool supported(int h, int w, int cin, int f) {
  if (f != 16 && f != 32) return false;
  const size_t smem = cin == 3 ? (f == 16 ? smem_bytes<3, 16>(h, w) : smem_bytes<3, 32>(h, w))
                               : (f == 16 ? smem_bytes<1, 16>(h, w) : smem_bytes<1, 32>(h, w));
  return smem <= 227 * 1024;
}

int fwd(const float* images, const float* kernel, const float* bias, void* out_planes, uint32_t* argmax, int64_t batch,
        int h, int w, int cin, int f, cudaStream_t st) {
  const int64_t cols = (int64_t)(h / 2) * (w / 2) * f;
  const pl::PlaneView pv = pl::plane_view(pl::format(), out_planes, batch, cols);
  if (cin == 3) return f == 16 ? launch<3, 16>(images, kernel, bias, pv, argmax, batch, h, w, st)
                               : launch<3, 32>(images, kernel, bias, pv, argmax, batch, h, w, st);
  return f == 16 ? launch<1, 16>(images, kernel, bias, pv, argmax, batch, h, w, st)
                 : launch<1, 32>(images, kernel, bias, pv, argmax, batch, h, w, st);
}

}  // namespace convtc
}  // namespace adn
