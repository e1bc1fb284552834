// K6: the SimpleCNN stem -- Conv2D(F, 3x3, "same") + bias + ReLU -> MaxPool2D(2, 2) -> Flatten -- fused into one
// forward kernel that writes the pooled features straight into the split-plane format the tcgen05 dense
// pipeline consumes (planes.cu), and one backward kernel for the kernel / bias gradients.
//
// Replaces the Keras layers of SimpleCNNBuilder.build_subnetwork in
//   adanet/examples/tutorials/customizing_adanet.ipynb (the `simple_cnn` subnetwork of BASELINE config 4):
//   x = Conv2D(filters=16, kernel_size=3, padding="same", activation="relu")(images)
//   x = MaxPool2D(pool_size=2, strides=2)(x);  x = Flatten()(x)            [TF/Keras, NHWC, HWIO kernel]
//
// Why SIMT fp32 and not tcgen05: the contraction is K = 9*Cin = 27 by N = F = 16 -- per example 0.44 MFMA against
// 12 KB of image read and ~37 KB of planes written, i.e. the kernel sits between the FP32-FMA rate and HBM, and
// an implicit-GEMM tile (K padded to 32, N=16) would leave the tensor pipe >90 % idle while adding an im2col
// stage.  Exact fp32 FMAs also keep the conv bit-comparable with the fp32 cross-check.
//
// Forward: one CTA per image (grid-stride), 256 threads, image staged zero-padded in shared memory with cp.async
// (double buffered: the next image lands while this one is computed); a thread owns one pooled pixel and 16
// filters at a time: 4 conv positions x 16 filters = 64 accumulators fed from the 4x4xCin patch in shared memory
// and float4 broadcast reads of the kernel (<= 128 registers: two CTAs per SM hide each other's latencies).  Epilogue: bias, ReLU, 2x2 max, hi/lo TF32 split, sign bits, and a
// 2-bit argmax per element for the backward.
// Backward: dK[ky,kx,c,f] = sum_{b,p} patch(b, argmax(b,p,f))[ky,kx,c] * g[b,p,f], db[f] = sum g, where g is the
// gradient w.r.t. the pooled features already masked by (pooled > 0) (the dX epilogue of the first dense layer
// applies the sign bits written here).  One thread per (channel, filter) pair holding the nine taps, images looped
// per CTA, per-CTA partials reduced in fixed order by a second kernel (deterministic).
#include <stdlib.h>

#include "common.cuh"
#include "plane_fmt.cuh"

namespace adn {

namespace convtc {
bool supported(int h, int w, int cin, int f);
int fwd(const float* images, const float* kernel, const float* bias, void* out_planes, uint32_t* argmax, int64_t batch,
        int h, int w, int cin, int f, cudaStream_t st);
}

namespace conv {

// ADN_CONV_PATH=simt forces the exact-fp32 SIMT forward (cross-check); default: tcgen05 implicit GEMM where supported
static bool use_tc() {      // read per call (host side, cheap): tests switch it at run time
  const char* e = getenv("ADN_CONV_PATH");
  return !(e && (e[0] == 's' || e[0] == 'S'));
}

static constexpr int FWD_THREADS = 256;
static constexpr int FC = 16;   // filters per accumulator chunk

__device__ __forceinline__ float rna_tf32(float v) {
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// image [H][W][CIN] (global) -> zero-padded [(H+2)][(W+2)][CIN] (shared); borders are zeroed once by the caller
template <int CIN>
__device__ __forceinline__ void stage_image(float* s_img, const float* img, int H, int W, int tid, int nthreads) {
  const int row = W * CIN;
  const int prow = (W + 2) * CIN;
  const int lane = tid & 31, nwarps = nthreads >> 5;
  for (int y = tid >> 5; y < H; y += nwarps) {          // a warp per image row: no per-element division
    const float* src = img + y * row;
    float* dst = s_img + (y + 1) * prow + CIN;
    for (int r = lane; r < row; r += 32) cp_async4(dst + r, src + r);
  }
}

template <int CIN>
__global__ void __launch_bounds__(FWD_THREADS, 2)
conv_stem_fwd_kernel(const float* __restrict__ images, const float* __restrict__ kernel, const float* __restrict__ bias,
                     const pl::PlaneView pv, unsigned int* ovf,
                     uint32_t* __restrict__ argmax, int64_t B, int H, int W, int F) {
  extern __shared__ __align__(16) float smem[];
  const int K = 9 * CIN;
  const int pimg = (H + 2) * (W + 2) * CIN;
  float* s_w = smem;                       // [K][F]
  float* s_b = s_w + K * F;                // [F]
  float* s_img0 = s_b + F;                 // two padded images
  const int tid = threadIdx.x;
  for (int i = tid; i < K * F; i += FWD_THREADS) s_w[i] = kernel[i];
  for (int i = tid; i < F; i += FWD_THREADS) s_b[i] = bias[i];
  for (int i = tid; i < 2 * pimg; i += FWD_THREADS) s_img0[i] = 0.f;
  __syncthreads();
  const int PH = H / 2, PW = W / 2, P = PH * PW;
  const int64_t img_elems = (int64_t)H * W * CIN;
  const int64_t words_per_row = (int64_t)P * F / 16;
  const int prow = (W + 2) * CIN;
  int64_t b = blockIdx.x;
  int buf = 0;
  if (b < B) stage_image<CIN>(s_img0, images + b * img_elems, H, W, tid, FWD_THREADS);
  cp_async_commit();
  for (; b < B; b += gridDim.x, buf ^= 1) {
    const int64_t nb = b + gridDim.x;
    if (nb < B) stage_image<CIN>(s_img0 + (buf ^ 1) * pimg, images + nb * img_elems, H, W, tid, FWD_THREADS);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const float* s_img = s_img0 + buf * pimg;
    for (int p = tid; p < P; p += FWD_THREADS) {
      const int py = p / PW, px = p - py * PW;
      // the 4x4xCIN input patch of this pooled pixel starts at padded coordinates (2py, 2px)
      const float* patch = s_img + (2 * py) * prow + (2 * px) * CIN;
      for (int f0 = 0; f0 < F; f0 += FC) {
        float acc[4][FC];
#pragma unroll
        for (int j = 0; j < FC; ++j) {
          const float bv = s_b[f0 + j];
          acc[0][j] = bv; acc[1][j] = bv; acc[2][j] = bv; acc[3][j] = bv;
        }
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int c = 0; c < CIN; ++c) {
              float w[FC];
              const float4* wp = reinterpret_cast<const float4*>(s_w + ((ky * 3 + kx) * CIN + c) * F + f0);
#pragma unroll
              for (int q = 0; q < FC / 4; ++q) {
                const float4 t = wp[q];
                w[4 * q] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w;
              }
#pragma unroll
              for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                for (int dx = 0; dx < 2; ++dx) {
                  const float v = patch[(dy + ky) * prow + (dx + kx) * CIN + c];
#pragma unroll
                  for (int j = 0; j < FC; ++j) acc[dy * 2 + dx][j] = fmaf(v, w[j], acc[dy * 2 + dx][j]);
                }
            }
        // bias is in; ReLU + 2x2 max (first maximum in scan order wins, as TF's MaxPoolGrad routes it)
        float outv[FC];
        uint32_t sign = 0u, arg = 0u;
#pragma unroll
        for (int j = 0; j < FC; ++j) {
          float m = acc[0][j];
          uint32_t a = 0u;
          if (acc[1][j] > m) { m = acc[1][j]; a = 1u; }
          if (acc[2][j] > m) { m = acc[2][j]; a = 2u; }
          if (acc[3][j] > m) { m = acc[3][j]; a = 3u; }
          m = fmaxf(m, 0.f);
          sign |= (m > 0.f) ? (1u << j) : 0u;
          arg |= a << (2 * j);
          outv[j] = m;
        }
        const int64_t col0 = (int64_t)p * F + f0;       // multiple of 16
#pragma unroll
        for (int q = 0; q < FC / 8; ++q) {
          float m8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) m8[e] = outv[8 * q + e];
          pl::plane_store8(pv, b, col0 + 8 * q, m8, ovf);
        }
        // sign bits: one uint32 per (32-column block, row); this thread owns one 16-bit half of it
        reinterpret_cast<uint16_t*>(pv.bits)[((col0 >> 5) * B + b) * 2 + ((col0 >> 4) & 1)] = (uint16_t)sign;
        argmax[b * words_per_row + (col0 >> 4)] = arg;
      }
    }
    __syncthreads();   // everyone is done with s_img[buf] before the next iteration's prefetch overwrites it
  }
}

// A thread owns one (channel c, filter f) pair and all nine taps: the gradient value and the arg-max word are read
// once per nine FMAs (the gather address depends on f through the arg-max, so taps are the only reuse there is).
// G groups of CIN*F threads split the pooled pixels of an image; their accumulators are summed in fixed order
// through shared memory once per CTA.
template <int CIN, int F>
__global__ void __launch_bounds__(1024)
conv_stem_bwd_kernel(const float* __restrict__ images, const uint32_t* __restrict__ argmax,
                     const float* __restrict__ dpooled, float* __restrict__ partials, int64_t B, int H, int W, int G) {
  extern __shared__ __align__(16) float smem[];
  const int K = 9 * CIN;
  const int PH = H / 2, PW = W / 2, P = PH * PW;
  const int pimg = (H + 2) * (W + 2) * CIN;
  const int prow = (W + 2) * CIN;
  // two staging sets {padded image, g [P*F], arg-max words [P*F/16]}: the next image is fetched under this one
  const int pimg4 = (pimg + 3) & ~3;
  const int set_floats = pimg4 + P * F + ((P * F / 16 + 3) & ~3);     // 16-byte aligned sets
  float* s_set0 = smem;
  float* s_red = smem + 2 * set_floats;                           // [G][K*F + F]
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < pimg; i += nt) { s_set0[i] = 0.f; s_set0[set_floats + i] = 0.f; }
  const int f = tid % F;
  const int c = (tid / F) % CIN;
  const int grp = tid / (F * CIN);
  const int wsel = f >> 4, sh = 2 * (f & 15);
  constexpr int fw = F / 16;
  float acc[9];
#pragma unroll
  for (int q = 0; q < 9; ++q) acc[q] = 0.f;
  float accb = 0.f;
  const int64_t img_elems = (int64_t)H * W * CIN;
  const int64_t cols = (int64_t)P * F;
  auto stage = [&](float* set, int64_t bb) {
    stage_image<CIN>(set, images + bb * img_elems, H, W, tid, nt);
    float* sg = set + pimg4;
    uint32_t* sa = reinterpret_cast<uint32_t*>(sg + P * F);
    for (int i = tid; i < (int)(cols / 4); i += nt) cp_async16(sg + 4 * i, dpooled + bb * cols + 4 * i);
    for (int i = tid; i < (int)(cols / 16); i += nt) cp_async4(sa + i, argmax + bb * (cols / 16) + i);
  };
  __syncthreads();
  int buf = 0;
  if ((int64_t)blockIdx.x < B) stage(s_set0, blockIdx.x);
  cp_async_commit();
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x, buf ^= 1) {
    const int64_t nb = b + gridDim.x;
    if (nb < B) stage(s_set0 + (buf ^ 1) * set_floats, nb);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const float* s_img = s_set0 + buf * set_floats;
    const float* s_g = s_img + pimg4;
    const uint32_t* s_arg = reinterpret_cast<const uint32_t*>(s_g + P * F);
    // groups stride the pooled pixels of a row; tap addresses are three row pointers + compile-time offsets
    for (int py = 0; py < PH; ++py) {
      const float* grow = s_g + (py * PW) * F + f;
      const uint32_t* arow = s_arg + (py * PW) * fw + wsel;
      const float* irow = s_img + (2 * py) * prow + c;
      for (int px = grp; px < PW; px += G) {
        const float g = grow[px * F];
        const uint32_t pos = (arow[px * fw] >> sh) & 3u;
        // padded coordinates of tap (0, 0) at the arg-max conv position (2py + dy, 2px + dx)
        const float* r0 = irow + (pos >> 1) * prow + (2 * px + (pos & 1u)) * CIN;
        const float* r1 = r0 + prow;
        const float* r2 = r1 + prow;
        acc[0] = fmaf(r0[0], g, acc[0]);
        acc[1] = fmaf(r0[CIN], g, acc[1]);
        acc[2] = fmaf(r0[2 * CIN], g, acc[2]);
        acc[3] = fmaf(r1[0], g, acc[3]);
        acc[4] = fmaf(r1[CIN], g, acc[4]);
        acc[5] = fmaf(r1[2 * CIN], g, acc[5]);
        acc[6] = fmaf(r2[0], g, acc[6]);
        acc[7] = fmaf(r2[CIN], g, acc[7]);
        acc[8] = fmaf(r2[2 * CIN], g, acc[8]);
        accb += g;
      }
    }
    __syncthreads();
  }
  // group-major partial sums -> fixed-order sum over groups -> this CTA's partial
  const int n_out = K * F + F;
  float* red = s_red + grp * n_out;
#pragma unroll
  for (int q = 0; q < 9; ++q) red[(q * CIN + c) * F + f] = acc[q];     // k = (ky*3+kx)*CIN + c
  if (c == 0) red[K * F + f] = accb;
  __syncthreads();
  float* mine = partials + (size_t)blockIdx.x * n_out;
  for (int i = tid; i < n_out; i += nt) {
    float s = 0.f;
    for (int q = 0; q < G; ++q) s += s_red[q * n_out + i];
    mine[i] = s;
  }
}

// one warp per output: lanes stride the per-CTA partials (fixed order), then a fixed shuffle tree -- deterministic,
// and n_part / 32 dependent adds per lane instead of n_part (a thread-per-output loop took 40 us for 592 partials)
__global__ void __launch_bounds__(256)
conv_stem_reduce_kernel(const float* __restrict__ partials, int n_part, int n_out, int kf, float* __restrict__ dkernel,
                        float* __restrict__ dbias) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // output index = global warp index
  const int lane = threadIdx.x & 31;
  if (i >= n_out) return;
  float s = 0.f;
  for (int q = lane; q < n_part; q += 32) s += partials[(size_t)q * n_out + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) {
    if (i < kf) dkernel[i] = s;
    else dbias[i - kf] = s;
  }
}

static constexpr size_t kMaxSmem = 200 * 1024;

// Dynamic shared-memory limits are raised ONCE here (adn_init): cudaFuncSetAttribute inside a stream capture can
// invalidate the capture (first use of a larger size while the engine records its CUDA graph).
int init() {
#define ADN_CONV_ATTR(K) ADN_CUDA(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem))
  ADN_CONV_ATTR(conv_stem_fwd_kernel<1>);
  ADN_CONV_ATTR(conv_stem_fwd_kernel<3>);
  ADN_CONV_ATTR((conv_stem_bwd_kernel<1, 16>)); ADN_CONV_ATTR((conv_stem_bwd_kernel<3, 16>));
  ADN_CONV_ATTR((conv_stem_bwd_kernel<1, 32>)); ADN_CONV_ATTR((conv_stem_bwd_kernel<3, 32>));
  ADN_CONV_ATTR((conv_stem_bwd_kernel<1, 48>)); ADN_CONV_ATTR((conv_stem_bwd_kernel<3, 48>));
  ADN_CONV_ATTR((conv_stem_bwd_kernel<1, 64>)); ADN_CONV_ATTR((conv_stem_bwd_kernel<3, 64>));
#undef ADN_CONV_ATTR
  return ADN_OK;
}

static int bwd_ctas(int64_t batch) {
  const int64_t cap = (int64_t)sm_count() * 4;
  return (int)(batch < cap ? batch : cap);
}

static int check_shape(const char* who, int64_t batch, int h, int w, int cin, int f) {
  if (batch < 1 || h < 2 || w < 2 || (h & 1) || (w & 1))
    return fail(ADN_ERR_INVALID, "%s: batch %lld, image %dx%d (height and width must be even and >= 2)", who,
                (long long)batch, h, w);
  if (cin != 1 && cin != 3) return fail(ADN_ERR_UNSUPPORTED, "%s: channels %d not in {1, 3}", who, cin);
  if (f < 16 || f > 64 || f % 16) return fail(ADN_ERR_UNSUPPORTED, "%s: filters %d not in {16, 32, 48, 64}", who, f);
  if ((int64_t)(h + 2) * (w + 2) * cin > 24 * 1024)
    return fail(ADN_ERR_UNSUPPORTED, "%s: image %dx%dx%d does not fit the shared-memory staging", who, h, w, cin);
  return ADN_OK;
}

int64_t bwd_workspace_bytes(int64_t batch, int cin, int f) {
  return (int64_t)bwd_ctas(batch) * (9 * cin * f + f) * (int64_t)sizeof(float);
}

}  // namespace conv
}  // namespace adn

using namespace adn;

extern "C" int adn_conv_stem_fwd(const float* images, const float* kernel, const float* bias, void* out_planes,
                                 uint32_t* argmax, int64_t batch, int height, int width, int channels, int filters,
                                 void* stream) {
  if (!images || !kernel || !bias || !out_planes || !argmax) return fail(ADN_ERR_INVALID, "adn_conv_stem_fwd: null pointer");
  if (int rc = conv::check_shape("adn_conv_stem_fwd", batch, height, width, channels, filters)) return rc;
  if (conv::use_tc() && convtc::supported(height, width, channels, filters))
    return convtc::fwd(images, kernel, bias, out_planes, argmax, batch, height, width, channels, filters, as_stream(stream));
  const int64_t cols = (int64_t)(height / 2) * (width / 2) * filters;
  const pl::PlaneView pv = pl::plane_view(pl::format(), out_planes, batch, cols);
  const int pimg = (height + 2) * (width + 2) * channels;
  const size_t smem = (size_t)(9 * channels * filters + filters + 2 * pimg) * sizeof(float);
  const int64_t cap = (int64_t)sm_count() * 2;
  const int grid = (int)(batch < cap ? batch : cap);
  if (smem > conv::kMaxSmem) return fail(ADN_ERR_UNSUPPORTED, "adn_conv_stem_fwd: %zu bytes of staging do not fit", smem);
  auto launch = [&](auto kern) -> int {
    kern<<<grid, conv::FWD_THREADS, smem, as_stream(stream)>>>(images, kernel, bias, pv, pl::overflow_flag(), argmax, batch,
                                                             height, width, filters);
    ADN_CHECK_LAUNCH("conv_stem_fwd");
    return ADN_OK;
  };
  return channels == 3 ? launch(conv::conv_stem_fwd_kernel<3>) : launch(conv::conv_stem_fwd_kernel<1>);
}

extern "C" int adn_conv_stem_bwd(const float* images, const uint32_t* argmax, const float* dpooled, float* dkernel,
                                 float* dbias, int64_t batch, int height, int width, int channels, int filters,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  if (!images || !argmax || !dpooled || !dkernel || !dbias) return fail(ADN_ERR_INVALID, "adn_conv_stem_bwd: null pointer");
  if (int rc = conv::check_shape("adn_conv_stem_bwd", batch, height, width, channels, filters)) return rc;
  const int64_t need = conv::bwd_workspace_bytes(batch, channels, filters);
  if (!workspace || workspace_bytes < need)
    return fail(ADN_ERR_WORKSPACE, "adn_conv_stem_bwd: workspace %lld < %lld bytes", (long long)workspace_bytes, (long long)need);
  const int kf = 9 * channels * filters;
  // G thread groups of channels*filters threads share the pooled pixels of an image (even, so threads % 32 == 0)
  int groups = (384 / (channels * filters)) & ~1;
  groups = groups < 2 ? 2 : (groups > 16 ? 16 : groups);
  const int threads = groups * channels * filters;
  const int grid = conv::bwd_ctas(batch);
  const int pimg = (height + 2) * (width + 2) * channels;
  const int64_t cols = (int64_t)(height / 2) * (width / 2) * filters;
  const size_t smem = (2 * ((size_t)((pimg + 3) & ~3) + cols + ((cols / 16 + 3) & ~(int64_t)3)) + (size_t)groups * (kf + filters)) * sizeof(float);
  if (smem > conv::kMaxSmem) return fail(ADN_ERR_UNSUPPORTED, "adn_conv_stem_bwd: %zu bytes of staging do not fit", smem);
  float* partials = static_cast<float*>(workspace);
  auto launch = [&](auto kern) -> int {
    kern<<<grid, threads, smem, as_stream(stream)>>>(images, argmax, dpooled, partials, batch, height, width, groups);
    ADN_CHECK_LAUNCH("conv_stem_bwd");
    return ADN_OK;
  };
  int rc = ADN_OK;
  switch (filters / 16 * 4 + channels) {      // filters in {16,32,48,64} x channels in {1,3}
    case 1 * 4 + 1: rc = launch(conv::conv_stem_bwd_kernel<1, 16>); break;
    case 1 * 4 + 3: rc = launch(conv::conv_stem_bwd_kernel<3, 16>); break;
    case 2 * 4 + 1: rc = launch(conv::conv_stem_bwd_kernel<1, 32>); break;
    case 2 * 4 + 3: rc = launch(conv::conv_stem_bwd_kernel<3, 32>); break;
    case 3 * 4 + 1: rc = launch(conv::conv_stem_bwd_kernel<1, 48>); break;
    case 3 * 4 + 3: rc = launch(conv::conv_stem_bwd_kernel<3, 48>); break;
    case 4 * 4 + 1: rc = launch(conv::conv_stem_bwd_kernel<1, 64>); break;
    default: rc = launch(conv::conv_stem_bwd_kernel<3, 64>); break;
  }
  if (rc) return rc;
  const int n_out = kf + filters;
  conv::conv_stem_reduce_kernel<<<(n_out * 32 + 255) / 256, 256, 0, as_stream(stream)>>>(partials, grid, n_out, kf, dkernel,
                                                                                   dbias);
  ADN_CHECK_LAUNCH("conv_stem_reduce");
  return ADN_OK;
}
