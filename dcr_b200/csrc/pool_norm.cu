// HBM-bound kernels between the tensor-core contractions of the descriptor networks.  Activations are NHWC bf16
// "planes" (1 plane = fast bf16 mode, 3 planes = hi/mid/lo split that carries fp32 precision); every kernel reads the
// sum of the planes, computes in fp32 and re-splits on store.  All channel counts are multiples of 8 so every access
// is a 16-byte vector.
//
// Reference ops replaced:
//   diff_retrieval.py:325-330  Resize(256)/CenterCrop(224)/ToTensor/Normalize            -> im2col_u8_kernel
//   embedding_search/utils.py:35-50 (ImageNet mean/std variant)                           -> im2col_u8_kernel
//   metrics/fid.py:104-110 + metrics/inception.py:152-153 (normalise twice)               -> im2col_u8_kernel (post affine)
//   torchvision resnet maxpool(3,2,1); inception max_pool2d(3,2)                          -> maxpool_kernel
//   metrics/inception.py:241,269,302 avg_pool2d(3,1,1,count_include_pad=False)            -> avgpool3_kernel
//   SSCD GeM pooling (p=3, eps=1e-6) [upstream, unverified]                               -> gem_kernel
//   metrics/inception.py adaptive_avg_pool2d((1,1))                                       -> global_avgpool_kernel
//   dino_vits.py:144-150,252 nn.LayerNorm(eps=1e-6)                                       -> layernorm_kernel
//   dino_vits.py:235-246 prepare_tokens (cls token + pos_embed)                           -> vit_tokens_kernel
#include <cuda_bf16.h>

#include <algorithm>

#include "dcr_internal.cuh"
#include "host_util.cuh"

namespace dcr {
namespace {

constexpr uint32_t kFull = 0xffffffffu;

__device__ __forceinline__ void load8(const __nv_bfloat16* base, long long plane_stride, int planes, size_t idx,
                                      float (&v)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = 0.f;
  for (int p = 0; p < planes; ++p) {
    const uint4 u = *reinterpret_cast<const uint4*>(base + p * plane_stride + idx);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] += __uint_as_float(w[j] << 16);
      v[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
    }
  }
}

__device__ __forceinline__ void store8(__nv_bfloat16* base, long long plane_stride, int planes, size_t idx,
                                       float (&v)[8]) {
  for (int p = 0; p < planes; ++p) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat16 a = __float2bfloat16_rn(v[2 * j]), b = __float2bfloat16_rn(v[2 * j + 1]);
      w[j] = static_cast<uint32_t>(__bfloat16_as_ushort(a)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b)) << 16);
      v[2 * j] -= __bfloat162float(a);
      v[2 * j + 1] -= __bfloat162float(b);
    }
    *reinterpret_cast<uint4*>(base + p * plane_stride + idx) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ---- uint8 HWC image -> normalised im2col matrix for the (3-channel) first convolution ------------------------
// out[m, k], m = (b, p, q) over the OHxOW output grid, k = (r*kw + s)*3 + c  (zero for k >= kh*kw*3 and for taps
// that fall into the zero padding).  value = post_scale * ((u8/255 - mean[c]) / std[c]) + post_shift.
struct Im2colU8Params {
  const uint8_t* img;
  const float* img_f32;   // kF32 kernels: fp32 NCHW [B,3,IH,IW], already transformed (ToTensor/Normalize done by the caller)
  int B, IH, IW, crop_y, crop_x, H, W;   // H, W: size after the centre crop
  int RH, RW;                            // network input size: == H, W, or the bilinearly resized crop (rscale != 0)
  float rscale;                          // float(1 / scale_factor) of utils_ret.py:676-698 `multi_scale`, 0 = no resizing
  int kh, kw, stride, pad, OH, OW, k_pad;
  float mean[3], std[3], post_scale, post_shift;
  __nv_bfloat16* out;
  long long out_plane_stride;
  int planes;
};

// K layout: k = r * RP + s * 3 + c with RP = ceil8(3 * KW) (each filter row padded to a multiple of 8 elements so
// that a thread owns whole 16-byte groups and every (s, c) index is a compile-time constant).  One thread per
// (output pixel, filter row): 3*KW contiguous image bytes -> RP normalised bf16 values.
// kF32: the input is the tensor the reference hands to `model(samples)` (utils_ret.py:751): fp32 NCHW, already
// normalised; only the optional post affine (FID's second 2x-1, inception.py:152-153) is applied.
template <int KW, bool kF32, bool kResize>
__global__ void __launch_bounds__(256) im2col_u8_kernel(const Im2colU8Params p) {
  constexpr int RP = (3 * KW + 7) / 8 * 8;
  // per-channel lookup table u8 -> normalised value, computed once per block with the reference's exact arithmetic
  // (ToTensor: u8/255, Normalize: (x-mean)/std, both fp32 with IEEE division), then the optional post affine
  __shared__ float lut[3][256];
  for (int i = threadIdx.x; i < 768; i += blockDim.x) {
    const int c = i >> 8, u = i & 255;
    const float val = (static_cast<float>(u) / 255.f - p.mean[c]) / p.std[c];
    lut[c][u] = p.post_scale * val + p.post_shift;
  }
  __syncthreads();
  const int rows_k = (p.k_pad + RP - 1) / RP;   // kh filter rows + zero rows up to k_pad (the last one may be partial)
  const long long total = static_cast<long long>(p.B) * p.OH * p.OW * rows_k;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i % rows_k);
    const long long m = i / rows_k;
    const int q = static_cast<int>(m % p.OW);
    const int pp = static_cast<int>((m / p.OW) % p.OH);
    const int b = static_cast<int>(m / (static_cast<long long>(p.OW) * p.OH));
    const int y = pp * p.stride - p.pad + r;           // in crop coordinates
    const int x0 = q * p.stride - p.pad;
    const bool row_ok = r < p.kh && y >= 0 && y < p.RH;
    const size_t plane = static_cast<size_t>(p.IH) * p.IW;
    const uint8_t* img = p.img + static_cast<size_t>(b) * p.IH * p.IW * 3;
    const float* imgf = p.img_f32 + static_cast<size_t>(b) * 3 * plane;
    // transformed value of channel c at crop coordinates (yy, xx)
    auto px = [&](int yy, int xx, int c) -> float {
      if constexpr (kF32) return fmaf(p.post_scale, imgf[c * plane + static_cast<size_t>(yy + p.crop_y) * p.IW + (xx + p.crop_x)], p.post_shift);
      else return lut[c][img[(static_cast<size_t>(yy + p.crop_y) * p.IW + (xx + p.crop_x)) * 3 + c]];
    };
    // bilinear source rows of the resized image (torch F.interpolate, align_corners=False, scale_factor given)
    int y0 = 0, y1 = 0;
    float ly = 0.f, hy = 1.f;
    if constexpr (kResize) {
      const float sy = fmaxf(p.rscale * (static_cast<float>(y) + 0.5f) - 0.5f, 0.f);
      y0 = min(static_cast<int>(sy), p.H - 1);
      y1 = y0 + (y0 < p.H - 1 ? 1 : 0);
      ly = sy - static_cast<float>(y0);
      hy = 1.f - ly;
    }
    __nv_bfloat16* dst = p.out + static_cast<size_t>(m) * p.k_pad + r * RP;
#pragma unroll
    for (int g = 0; g < RP / 8; ++g) {
      if (r * RP + g * 8 >= p.k_pad) break;   // partial last zero row (k_pad is a multiple of 8, not always of RP)
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int j = g * 8 + e;          // compile-time after unrolling
        const int s = j / 3, c = j % 3;
        float val = 0.f;
        if (j < 3 * KW && row_ok && x0 + s >= 0 && x0 + s < p.RW) {
          if constexpr (kResize) {
            const float sx = fmaxf(p.rscale * (static_cast<float>(x0 + s) + 0.5f) - 0.5f, 0.f);
            const int xa = min(static_cast<int>(sx), p.W - 1);
            const int xb = xa + (xa < p.W - 1 ? 1 : 0);
            const float lx = sx - static_cast<float>(xa), hx = 1.f - lx;
            val = hy * (hx * px(y0, xa, c) + lx * px(y0, xb, c)) + ly * (hx * px(y1, xa, c) + lx * px(y1, xb, c));
          } else {
            val = px(y, x0 + s, c);
          }
        }
        v[e] = val;
      }
      store8(dst, p.out_plane_stride, p.planes, g * 8, v);
    }
  }
}

// ---- space-to-depth stem input (7x7 / stride 2 / pad 3 first convolution of the ResNet trunk) ----------------------
// Z[b, u, v, (i*2+j)*3 + c] = xn[2u + i - 3, 2v + j - 3, c]  (zero outside the image), channels 12..15 = 0, with
// xn the normalised crop.  A 7x7/2 convolution of xn equals a 4x4/1 convolution of Z (weights regrouped on the host),
// which the GEMM kernel reads through an overlapping-window tensor map -- no im2col matrix in HBM.
// Optional bilinear down-scaling of the normalised crop first (utils_ret.py:676-698 `multi_scale`:
// F.interpolate(x, scale_factor=s, mode='bilinear', align_corners=False)): xn is then the [RH, RW] resized image,
// sampled with torch's arithmetic (source index = rscale * (dst + 0.5) - 0.5 clamped at 0, rscale = float(1 / s)).
struct StemS2dParams {
  const uint8_t* img;
  const float* img_f32;   // kF32 kernels: fp32 NCHW [B,3,IH,IW], already transformed
  int B, IH, IW, crop_y, crop_x, H, W, U, V;
  int RH, RW;        // size of xn (== H, W without resizing)
  float rscale;      // 0 = no resizing
  float mean[3], std[3], post_scale, post_shift;
  __nv_bfloat16* out;
  long long out_plane_stride;
  int planes;
};

template <bool kResize, bool kF32>
__global__ void __launch_bounds__(256) stem_s2d_u8_kernel(const StemS2dParams p) {
  __shared__ float lut[3][256];
  for (int i = threadIdx.x; i < 768; i += blockDim.x) {
    const int c = i >> 8, u = i & 255;
    const float val = (static_cast<float>(u) / 255.f - p.mean[c]) / p.std[c];   // ToTensor + Normalize, IEEE fp32
    lut[c][u] = p.post_scale * val + p.post_shift;
  }
  __syncthreads();
  const long long total = static_cast<long long>(p.B) * p.U * p.V;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(idx % p.V);
    const int u = static_cast<int>((idx / p.V) % p.U);
    const int b = static_cast<int>(idx / (static_cast<long long>(p.V) * p.U));
    const uint8_t* img = p.img + static_cast<size_t>(b) * p.IH * p.IW * 3;
    const size_t plane = static_cast<size_t>(p.IH) * p.IW;
    const float* imgf = p.img_f32 + static_cast<size_t>(b) * 3 * plane;
    // normalised value of channel c at crop coordinates (yy, xx)
    auto px = [&](int yy, int xx, int c) -> float {
      if constexpr (kF32) return fmaf(p.post_scale, imgf[c * plane + static_cast<size_t>(yy + p.crop_y) * p.IW + (xx + p.crop_x)], p.post_shift);
      else return lut[c][img[(static_cast<size_t>(yy + p.crop_y) * p.IW + (xx + p.crop_x)) * 3 + c]];
    };
    float z[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) z[e] = 0.f;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int y = 2 * u + i - 3;
      if (y < 0 || y >= p.RH) continue;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int x = 2 * v + j - 3;
        if (x < 0 || x >= p.RW) continue;
        if constexpr (!kResize) {
#pragma unroll
          for (int c = 0; c < 3; ++c) z[(i * 2 + j) * 3 + c] = px(y, x, c);
        } else {
          const float sy = fmaxf(p.rscale * (static_cast<float>(y) + 0.5f) - 0.5f, 0.f);
          const float sx = fmaxf(p.rscale * (static_cast<float>(x) + 0.5f) - 0.5f, 0.f);
          const int y0 = static_cast<int>(sy), x0 = static_cast<int>(sx);
          const int y1 = y0 + (y0 < p.H - 1 ? 1 : 0), x1 = x0 + (x0 < p.W - 1 ? 1 : 0);
          const float ly = sy - static_cast<float>(y0), lx = sx - static_cast<float>(x0);
          const float hy = 1.f - ly, hx = 1.f - lx;
#pragma unroll
          for (int c = 0; c < 3; ++c)
            z[(i * 2 + j) * 3 + c] = hy * (hx * px(y0, x0, c) + lx * px(y0, x1, c)) +
                                     ly * (hx * px(y1, x0, c) + lx * px(y1, x1, c));
        }
      }
    }
    float lo[8], hi[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      lo[e] = z[e];
      hi[e] = z[8 + e];
    }
    store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(idx) * 16, lo);
    store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(idx) * 16 + 8, hi);
  }
}

// ---- pooling -------------------------------------------------------------------------------------------------
struct PoolParams {
  const __nv_bfloat16* in;
  long long in_plane_stride;
  __nv_bfloat16* out;
  long long out_plane_stride;
  int planes;
  int B, H, W, C, k, stride, pad, OH, OW, ld_out, out_col_off;
};

template <bool kMax>
__global__ void pool_kernel(const PoolParams p) {
  const int cg = p.C / 8;
  const long long total = static_cast<long long>(p.B) * p.OH * p.OW * cg;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg);
    const long long m = i / cg;
    const int q = static_cast<int>(m % p.OW);
    const int pp = static_cast<int>((m / p.OW) % p.OH);
    const int b = static_cast<int>(m / (static_cast<long long>(p.OW) * p.OH));
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = kMax ? -INFINITY : 0.f;
    int cnt = 0;
    for (int r = 0; r < p.k; ++r) {
      const int y = pp * p.stride - p.pad + r;
      if (y < 0 || y >= p.H) continue;
      for (int s = 0; s < p.k; ++s) {
        const int x = q * p.stride - p.pad + s;
        if (x < 0 || x >= p.W) continue;
        float v[8];
        load8(p.in, p.in_plane_stride, p.planes, ((static_cast<size_t>(b) * p.H + y) * p.W + x) * p.C + c8 * 8, v);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = kMax ? fmaxf(acc[e], v[e]) : acc[e] + v[e];
        ++cnt;
      }
    }
    if (!kMax) {
      // count_include_pad=False: divide by the number of in-bounds taps
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] = acc[e] / static_cast<float>(cnt);
    }
    store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(m) * p.ld_out + p.out_col_off + c8 * 8, acc);
  }
}

// Single-plane 3x3 average pool, count_include_pad = False (the patched pools of the FID Inception blocks,
// metrics/inception.py:241,269,302): nine clamped 16-byte loads in flight per thread, fp32 sum of the in-bounds taps in the
// generic kernel's order (bit-identical results), one division.  The generic kernel walked the taps serially: 1.4 ms of a
// 5.5 ms Inception forward at batch 128 (profiles/r02_layers_inception.txt) for data HBM moves in ~0.15 ms.
__global__ void __launch_bounds__(256) avgpool3_bf16_kernel(const PoolParams p) {
  const int cg = p.C / 8;
  const long long total = static_cast<long long>(p.B) * p.OH * p.OW * cg;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg);
    const long long m = i / cg;
    const int q = static_cast<int>(m % p.OW);
    const int pp = static_cast<int>((m / p.OW) % p.OH);
    const int b = static_cast<int>(m / (static_cast<long long>(p.OW) * p.OH));
    const int y0 = pp * p.stride - p.pad, x0 = q * p.stride - p.pad;
    const __nv_bfloat16* img = p.in + static_cast<size_t>(b) * p.H * p.W * p.C + c8 * 8;
    uint4 v[9];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const __nv_bfloat16* row = img + static_cast<size_t>(min(max(y0 + r, 0), p.H - 1)) * p.W * p.C;
#pragma unroll
      for (int s = 0; s < 3; ++s)
        v[r * 3 + s] = __ldg(reinterpret_cast<const uint4*>(row + static_cast<size_t>(min(max(x0 + s, 0), p.W - 1)) * p.C));
    }
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    int cnt = 0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int y = y0 + r, x = x0 + s;
        if (y >= 0 && y < p.H && x >= 0 && x < p.W) {
          const uint32_t w[4] = {v[r * 3 + s].x, v[r * 3 + s].y, v[r * 3 + s].z, v[r * 3 + s].w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc[2 * j] += __uint_as_float(w[j] << 16);
            acc[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
          }
          ++cnt;
        }
      }
    }
    const float fc = static_cast<float>(cnt);
    uint4 o;
    __nv_bfloat162 t0 = __floats2bfloat162_rn(acc[0] / fc, acc[1] / fc), t1 = __floats2bfloat162_rn(acc[2] / fc, acc[3] / fc);
    __nv_bfloat162 t2 = __floats2bfloat162_rn(acc[4] / fc, acc[5] / fc), t3 = __floats2bfloat162_rn(acc[6] / fc, acc[7] / fc);
    o.x = *reinterpret_cast<uint32_t*>(&t0); o.y = *reinterpret_cast<uint32_t*>(&t1);
    o.z = *reinterpret_cast<uint32_t*>(&t2); o.w = *reinterpret_cast<uint32_t*>(&t3);
    *reinterpret_cast<uint4*>(p.out + static_cast<size_t>(m) * p.ld_out + p.out_col_off + c8 * 8) = o;
  }
}

// Single-plane 3x3 max pool (any stride / padding): the fast-mode path of the ResNet stem and the three Inception
// reductions.  bf16 maxima are taken directly on the packed pairs (the maximum of bf16 values is exact), the nine
// 16-byte loads are issued unconditionally from clamped coordinates (out-of-range taps are masked with -inf after the
// load) so they are all in flight together, and each thread produces two horizontally adjacent outputs so that the
// shared middle column of their windows is loaded once.
__global__ void __launch_bounds__(256) maxpool3_bf16_kernel(const PoolParams p) {
  const int cg = p.C / 8;
  const int OW2 = (p.OW + 1) / 2;
  const long long total = static_cast<long long>(p.B) * p.OH * OW2 * cg;
  const __nv_bfloat162 ninf = __floats2bfloat162_rn(-INFINITY, -INFINITY);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg);
    const long long m2 = i / cg;
    const int q0 = static_cast<int>(m2 % OW2) * 2;
    const int pp = static_cast<int>((m2 / OW2) % p.OH);
    const int b = static_cast<int>(m2 / (static_cast<long long>(OW2) * p.OH));
    const int y0 = pp * p.stride - p.pad, x0 = q0 * p.stride - p.pad;
    const int ncols = 3 + p.stride;                 // columns covered by the two windows (<= 5 for stride <= 2)
    __nv_bfloat162 a0[4], a1[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) a0[e] = a1[e] = ninf;
    const __nv_bfloat16* img = p.in + static_cast<size_t>(b) * p.H * p.W * p.C + c8 * 8;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int y = y0 + r;
      const bool yok = y >= 0 && y < p.H;
      const __nv_bfloat16* row = img + static_cast<size_t>(min(max(y, 0), p.H - 1)) * p.W * p.C;
      uint4 v[5];
#pragma unroll
      for (int s = 0; s < 5; ++s) {
        const int x = x0 + s;
        v[s] = __ldg(reinterpret_cast<const uint4*>(row + static_cast<size_t>(min(max(x, 0), p.W - 1)) * p.C));
      }
#pragma unroll
      for (int s = 0; s < 5; ++s) {
        const int x = x0 + s;
        const bool ok = yok && x >= 0 && x < p.W && s < ncols;
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v[s]);
        const bool in0 = ok && s < 3, in1 = ok && s >= p.stride && s < p.stride + 3;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (in0) a0[e] = __hmax2(a0[e], h[e]);
          if (in1) a1[e] = __hmax2(a1[e], h[e]);
        }
      }
    }
    const size_t m = (static_cast<size_t>(b) * p.OH + pp) * p.OW + q0;
    __nv_bfloat16* o = p.out + m * p.ld_out + p.out_col_off + c8 * 8;
    *reinterpret_cast<uint4*>(o) = *reinterpret_cast<const uint4*>(a0);
    if (q0 + 1 < p.OW) *reinterpret_cast<uint4*>(o + p.ld_out) = *reinterpret_cast<const uint4*>(a1);
  }
}

// ---- GeM / global average over the spatial positions of one image --------------------------------------------
// grid = (B, C/8 / 32 rounded up); each thread owns one 8-channel group of one image and walks HW positions.
struct ReduceHWParams {
  const __nv_bfloat16* in;
  long long in_plane_stride;
  int planes, B, HW, C;
  float p_exp, eps;          // GeM only
  __nv_bfloat16* out;        // planes [B, C] or null
  long long out_plane_stride;
  float* out_f32;            // [B, C] or null
};

// block = 64 channel groups x kSlices position slices: every thread streams HW / kSlices positions of its 8 channels
// (independent 16-byte loads, several in flight), the slices meet in shared memory.  (One thread per channel group walked
// all HW positions serially before: 41 us for the 51 MB layer4 output of a ResNet-50 batch.)
constexpr int kRedSlices = 4;
// kCube: GeM with p = 3 (the SSCD head): t*t*t and cbrtf; the general exponent keeps powf out of this instantiation (inlined
// into the unrolled loop it made the kernel instruction-fetch bound: 39 us, 26 % of the warp samples on `no_inst`).
template <bool kGem, bool kCube>
__global__ void __launch_bounds__(64 * kRedSlices) reduce_hw_kernel(const ReduceHWParams p) {
  __shared__ float part[kRedSlices][64][8];
  const int cg = p.C / 8;
  const int b = blockIdx.x;
  const int tc = threadIdx.x & 63, slice = threadIdx.x >> 6;
  for (int c0 = blockIdx.y * 64; c0 < cg; c0 += gridDim.y * 64) {
    const int c8 = c0 + tc;
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    if (c8 < cg) {
#pragma unroll 4
      for (int i = slice; i < p.HW; i += kRedSlices) {
        float v[8];
        load8(p.in, p.in_plane_stride, p.planes, (static_cast<size_t>(b) * p.HW + i) * p.C + c8 * 8, v);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          if (kGem) {
            const float t = fmaxf(v[e], p.eps);
            acc[e] += kCube ? t * t * t : powf(t, p.p_exp);
          } else {
            acc[e] += v[e];
          }
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) part[slice][tc][e] = acc[e];
    __syncthreads();
    if (slice == 0 && c8 < cg) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float t = part[0][tc][e];
#pragma unroll
        for (int sl = 1; sl < kRedSlices; ++sl) t += part[sl][tc][e];   // fixed order: deterministic
        t = t / static_cast<float>(p.HW);
        if (kGem) t = kCube ? cbrtf(t) : powf(t, 1.f / p.p_exp);
        acc[e] = t;
      }
      if (p.out_f32) {
#pragma unroll
        for (int e = 0; e < 8; ++e) p.out_f32[static_cast<size_t>(b) * p.C + c8 * 8 + e] = acc[e];
      }
      if (p.out) store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(b) * p.C + c8 * 8, acc);
    }
    __syncthreads();
  }
}

// ---- LayerNorm over the last dim, one warp per row -------------------------------------------------------------
struct LayerNormParams {
  const __nv_bfloat16* in;
  long long in_plane_stride;
  int planes, rows, C;
  long long in_row_stride;    // elements between consecutive input rows (C for all rows, T*C for the CLS rows only)
  const float* gamma;
  const float* beta;
  float eps;
  __nv_bfloat16* out;         // planes [rows, C] or null
  long long out_plane_stride;
  float* out_f32;             // [rows, C] or null
};

// Single-plane fast path for C = kChunks * 128 (384, 512, 768, 1024): HALF a warp per row, kChunks 16-byte loads per lane
// all in flight at once (balanced: the generic kernel gives C = 384 to 32 + 16 lanes), gamma / beta held in registers across
// the rows a half-warp walks, 4-step reductions.  The generic kernel ran at ~2 TB/s (37 us for the 50k x 384 rows of a
// ViT-S/16 batch); this one is a pure stream.
template <int kChunks>
__global__ void __launch_bounds__(256) layernorm_fast_kernel(const LayerNormParams p) {
  const int lane16 = threadIdx.x & 15;
  const uint32_t hmask = 0xffffu << (threadIdx.x & 16);                   // this half-warp's lanes (the halves may run out of rows separately)
  const int hw = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;           // global half-warp index
  const int n_hw = (gridDim.x * blockDim.x) >> 4;
  float gm[kChunks][8], bt[kChunks][8];
#pragma unroll
  for (int g = 0; g < kChunks; ++g) {
    const int c = (g * 16 + lane16) * 8;
    const float4 g0 = *reinterpret_cast<const float4*>(p.gamma + c), g1 = *reinterpret_cast<const float4*>(p.gamma + c + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(p.beta + c), b1 = *reinterpret_cast<const float4*>(p.beta + c + 4);
    gm[g][0] = g0.x; gm[g][1] = g0.y; gm[g][2] = g0.z; gm[g][3] = g0.w; gm[g][4] = g1.x; gm[g][5] = g1.y; gm[g][6] = g1.z; gm[g][7] = g1.w;
    bt[g][0] = b0.x; bt[g][1] = b0.y; bt[g][2] = b0.z; bt[g][3] = b0.w; bt[g][4] = b1.x; bt[g][5] = b1.y; bt[g][6] = b1.z; bt[g][7] = b1.w;
  }
  constexpr float kInvC = 1.f / static_cast<float>(kChunks * 128);
  for (int row = hw; row < p.rows; row += n_hw) {
    const __nv_bfloat16* src = p.in + static_cast<size_t>(row) * p.in_row_stride;
    uint4 raw[kChunks];
#pragma unroll
    for (int g = 0; g < kChunks; ++g) raw[g] = *reinterpret_cast<const uint4*>(src + (g * 16 + lane16) * 8);
    float v[kChunks][8];
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < kChunks; ++g) {
      const uint32_t w[4] = {raw[g].x, raw[g].y, raw[g].z, raw[g].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[g][2 * j] = __uint_as_float(w[j] << 16);
        v[g][2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
        s += v[g][2 * j] + v[g][2 * j + 1];
      }
    }
#pragma unroll
    for (int off = 8; off > 0; off >>= 1) s += __shfl_xor_sync(hmask, s, off);    // within the half-warp
    const float mean = s * kInvC;
    float ss = 0.f;
#pragma unroll
    for (int g = 0; g < kChunks; ++g)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d = v[g][e] - mean;
        ss += d * d;
      }
#pragma unroll
    for (int off = 8; off > 0; off >>= 1) ss += __shfl_xor_sync(hmask, ss, off);
    const float rstd = 1.f / sqrtf(ss * kInvC + p.eps);                             // biased variance, as nn.LayerNorm
#pragma unroll
    for (int g = 0; g < kChunks; ++g) {
      float y[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) y[e] = (v[g][e] - mean) * rstd * gm[g][e] + bt[g][e];
      const size_t o = static_cast<size_t>(row) * (kChunks * 128) + (g * 16 + lane16) * 8;
      if (p.out_f32) {
        *reinterpret_cast<float4*>(p.out_f32 + o) = make_float4(y[0], y[1], y[2], y[3]);
        *reinterpret_cast<float4*>(p.out_f32 + o + 4) = make_float4(y[4], y[5], y[6], y[7]);
      }
      if (p.out) {
        uint4 q;
        __nv_bfloat162 t0 = __floats2bfloat162_rn(y[0], y[1]), t1 = __floats2bfloat162_rn(y[2], y[3]);
        __nv_bfloat162 t2 = __floats2bfloat162_rn(y[4], y[5]), t3 = __floats2bfloat162_rn(y[6], y[7]);
        q.x = *reinterpret_cast<uint32_t*>(&t0); q.y = *reinterpret_cast<uint32_t*>(&t1);
        q.z = *reinterpret_cast<uint32_t*>(&t2); q.w = *reinterpret_cast<uint32_t*>(&t3);
        *reinterpret_cast<uint4*>(p.out + o) = q;
      }
    }
  }
}

__global__ void layernorm_kernel(const LayerNormParams p) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  constexpr int kMaxGroups = 4;   // C <= 32 lanes * 4 groups * 8 = 1024
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < p.rows; row += gridDim.x * wpb) {
    const size_t base = static_cast<size_t>(row) * p.in_row_stride;
    float v[kMaxGroups][8];
    float s = 0.f;
    const int cg = p.C / 8;
#pragma unroll
    for (int g = 0; g < kMaxGroups; ++g) {
      const int c8 = lane + g * 32;
      if (c8 < cg) {
        load8(p.in, p.in_plane_stride, p.planes, base + c8 * 8, v[g]);
#pragma unroll
        for (int e = 0; e < 8; ++e) s += v[g][e];
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(kFull, s, off);
    const float mean = s / static_cast<float>(p.C);
    float ss = 0.f;
#pragma unroll
    for (int g = 0; g < kMaxGroups; ++g) {
      const int c8 = lane + g * 32;
      if (c8 < cg) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float d = v[g][e] - mean;
          ss += d * d;
        }
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(kFull, ss, off);
    const float rstd = 1.f / sqrtf(ss / static_cast<float>(p.C) + p.eps);   // biased variance, as nn.LayerNorm
#pragma unroll
    for (int g = 0; g < kMaxGroups; ++g) {
      const int c8 = lane + g * 32;
      if (c8 < cg) {
        const float4 g0 = *reinterpret_cast<const float4*>(p.gamma + c8 * 8);
        const float4 g1 = *reinterpret_cast<const float4*>(p.gamma + c8 * 8 + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(p.beta + c8 * 8);
        const float4 b1 = *reinterpret_cast<const float4*>(p.beta + c8 * 8 + 4);
        const float gm[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bt[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        float y[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) y[e] = (v[g][e] - mean) * rstd * gm[e] + bt[e];
        if (p.out_f32) {
          float* o = p.out_f32 + static_cast<size_t>(row) * p.C + c8 * 8;
          *reinterpret_cast<float4*>(o) = make_float4(y[0], y[1], y[2], y[3]);
          *reinterpret_cast<float4*>(o + 4) = make_float4(y[4], y[5], y[6], y[7]);
        }
        if (p.out) store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(row) * p.C + c8 * 8, y);
      }
    }
  }
}

// ---- ViT token assembly: tokens[b,0] = cls + pos[0]; tokens[b,1+i] = patch[b,i] + pos[1+i] ---------------------
struct VitTokensParams {
  const __nv_bfloat16* patch;   // planes [B*NP, C]
  long long patch_plane_stride;
  const float* cls;             // [C]
  const float* pos;             // [(NP+1), C]
  __nv_bfloat16* out;           // planes [B*(NP+1), C]
  long long out_plane_stride;
  int planes, B, NP, C;
};

__global__ void vit_tokens_kernel(const VitTokensParams p) {
  const int cg = p.C / 8;
  const long long total = static_cast<long long>(p.B) * (p.NP + 1) * cg;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg);
    const long long row = i / cg;
    const int t = static_cast<int>(row % (p.NP + 1));
    const int b = static_cast<int>(row / (p.NP + 1));
    float v[8];
    if (t == 0) {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = p.cls[c8 * 8 + e];
    } else {
      load8(p.patch, p.patch_plane_stride, p.planes, (static_cast<size_t>(b) * p.NP + (t - 1)) * p.C + c8 * 8, v);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] += p.pos[static_cast<size_t>(t) * p.C + c8 * 8 + e];
    store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(row) * p.C + c8 * 8, v);
  }
}

// ---- token embedding: planes[b*T + t, :] = table[ids[b, t], :] + pos[t, :]   (CLIP text tower input) ---------------------
struct EmbedParams {
  const int* ids;
  const float* table;
  const float* pos;
  __nv_bfloat16* out;
  long long out_plane_stride;
  int planes, B, T, C, vocab;
};
__global__ void embed_tokens_kernel(const EmbedParams p) {
  const int cg = p.C / 8;
  const long long total = static_cast<long long>(p.B) * p.T * cg;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg);
    const long long row = i / cg;
    const int t = static_cast<int>(row % p.T);
    int id = p.ids[row];
    id = id < 0 ? 0 : (id >= p.vocab ? p.vocab - 1 : id);
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e)
      v[e] = p.table[static_cast<size_t>(id) * p.C + c8 * 8 + e] + p.pos[static_cast<size_t>(t) * p.C + c8 * 8 + e];
    store8(p.out, p.out_plane_stride, p.planes, static_cast<size_t>(row) * p.C + c8 * 8, v);
  }
}

int grid_for(long long work_items, int block, int num_sms) {
  long long blocks = (work_items + block - 1) / block;
  return static_cast<int>(std::min<long long>(blocks, static_cast<long long>(num_sms) * 16));
}

}  // namespace

int im2col_u8(const uint8_t* img, int B, int IH, int IW, int crop_y, int crop_x, int H, int W, int kh, int kw,
              int stride, int pad, int k_pad, const float* mean3, const float* std3, float post_scale,
              float post_shift, __nv_bfloat16* out, long long out_plane_stride, int planes, cudaStream_t stream,
              const float* img_f32, int RH, int RW, float rscale) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  const int rp = (3 * kw + 7) / 8 * 8;
  DCR_REQUIRE(k_pad % 8 == 0 && k_pad >= kh * rp, "im2col_u8: k_pad %d must be a multiple of 8 and >= %d", k_pad, kh * rp);
  DCR_REQUIRE(kw == 3 || kw == 7 || kw == 8 || kw == 14 || kw == 16, "im2col_u8: filter width %d not instantiated (3, 7, 8, 14, 16)", kw);
  DCR_REQUIRE(crop_y >= 0 && crop_x >= 0 && crop_y + H <= IH && crop_x + W <= IW, "im2col_u8: crop outside image");
  Im2colU8Params p;
  p.img = img; p.img_f32 = img_f32; p.B = B; p.IH = IH; p.IW = IW; p.crop_y = crop_y; p.crop_x = crop_x; p.H = H; p.W = W;
  p.kh = kh; p.kw = kw; p.stride = stride; p.pad = pad;
  if (rscale == 0.f) { RH = H; RW = W; }
  DCR_REQUIRE(RH >= kh && RW >= kw, "im2col_u8: network input %d x %d smaller than the filter", RH, RW);
  p.RH = RH; p.RW = RW; p.rscale = rscale;
  p.OH = (RH + 2 * pad - kh) / stride + 1;
  p.OW = (RW + 2 * pad - kw) / stride + 1;
  p.k_pad = k_pad;
  for (int c = 0; c < 3; ++c) { p.mean[c] = mean3[c]; p.std[c] = std3[c]; }
  p.post_scale = post_scale; p.post_shift = post_shift;
  p.out = out; p.out_plane_stride = out_plane_stride; p.planes = planes;
  if (B == 0) return 0;
  const long long total = static_cast<long long>(B) * p.OH * p.OW * ((k_pad + rp - 1) / rp);
  const int grid = grid_for(total, 256, di->num_sms);
#define DCR_IM2COL(KWv)                                                                             \
  do {                                                                                              \
    if (img_f32) {                                                                                  \
      if (rscale == 0.f) im2col_u8_kernel<KWv, true, false><<<grid, 256, 0, stream>>>(p);           \
      else im2col_u8_kernel<KWv, true, true><<<grid, 256, 0, stream>>>(p);                          \
    } else {                                                                                        \
      if (rscale == 0.f) im2col_u8_kernel<KWv, false, false><<<grid, 256, 0, stream>>>(p);          \
      else im2col_u8_kernel<KWv, false, true><<<grid, 256, 0, stream>>>(p);                         \
    }                                                                                               \
  } while (0)
  if (kw == 7) DCR_IM2COL(7);
  else if (kw == 3) DCR_IM2COL(3);
  else if (kw == 8) DCR_IM2COL(8);
  else if (kw == 14) DCR_IM2COL(14);
  else DCR_IM2COL(16);
#undef DCR_IM2COL
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int embed_tokens(const int* ids, int B, int T, int C, const float* table, int vocab, const float* pos, __nv_bfloat16* out,
                 long long out_plane_stride, int planes, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(ids && table && pos && out && C % 8 == 0 && T >= 1 && vocab >= 1, "embed_tokens: bad arguments");
  if (B == 0) return 0;
  EmbedParams p;
  p.ids = ids; p.table = table; p.pos = pos; p.out = out; p.out_plane_stride = out_plane_stride;
  p.planes = planes; p.B = B; p.T = T; p.C = C; p.vocab = vocab;
  embed_tokens_kernel<<<grid_for(static_cast<long long>(B) * T * (C / 8), 256, di->num_sms), 256, 0, stream>>>(p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int stem_s2d_u8(const uint8_t* img, int B, int IH, int IW, int crop_y, int crop_x, int H, int W, const float* mean3,
                const float* std3, float post_scale, float post_shift, __nv_bfloat16* out, long long out_plane_stride,
                int planes, cudaStream_t stream, int RH, int RW, float rscale, const float* img_f32) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(crop_y >= 0 && crop_x >= 0 && crop_y + H <= IH && crop_x + W <= IW, "stem_s2d_u8: crop outside image");
  if (rscale == 0.f) { RH = H; RW = W; }
  DCR_REQUIRE(RH >= 2 && RW >= 2 && RH % 2 == 0 && RW % 2 == 0, "stem_s2d_u8: network input size must be even (%d x %d)", RH, RW);
  StemS2dParams p;
  p.img = img; p.img_f32 = img_f32; p.B = B; p.IH = IH; p.IW = IW; p.crop_y = crop_y; p.crop_x = crop_x; p.H = H; p.W = W;
  p.RH = RH; p.RW = RW; p.rscale = rscale;
  p.U = (RH + 6) / 2; p.V = (RW + 6) / 2;
  for (int c = 0; c < 3; ++c) { p.mean[c] = mean3[c]; p.std[c] = std3[c]; }
  p.post_scale = post_scale; p.post_shift = post_shift;
  p.out = out; p.out_plane_stride = out_plane_stride; p.planes = planes;
  if (B == 0) return 0;
  const long long total = static_cast<long long>(B) * p.U * p.V;
  const int grid = grid_for(total, 256, di->num_sms);
  if (img_f32) {
    if (rscale == 0.f) stem_s2d_u8_kernel<false, true><<<grid, 256, 0, stream>>>(p);
    else stem_s2d_u8_kernel<true, true><<<grid, 256, 0, stream>>>(p);
  } else {
    if (rscale == 0.f) stem_s2d_u8_kernel<false, false><<<grid, 256, 0, stream>>>(p);
    else stem_s2d_u8_kernel<true, false><<<grid, 256, 0, stream>>>(p);
  }
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int pool2d(bool is_max, const __nv_bfloat16* in, long long in_plane_stride, __nv_bfloat16* out,
           long long out_plane_stride, int planes, int B, int H, int W, int C, int k, int stride, int pad, int ld_out,
           int out_col_off, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(C % 8 == 0 && ld_out % 8 == 0 && out_col_off % 8 == 0, "pool2d: channel counts must be multiples of 8");
  PoolParams p;
  p.in = in; p.in_plane_stride = in_plane_stride; p.out = out; p.out_plane_stride = out_plane_stride;
  p.planes = planes; p.B = B; p.H = H; p.W = W; p.C = C; p.k = k; p.stride = stride; p.pad = pad;
  p.OH = (H + 2 * pad - k) / stride + 1;
  p.OW = (W + 2 * pad - k) / stride + 1;
  p.ld_out = ld_out; p.out_col_off = out_col_off;
  if (B == 0) return 0;
  const long long total = static_cast<long long>(B) * p.OH * p.OW * (C / 8);
  if (is_max && planes == 1 && k == 3 && stride <= 2 && !tuning_flag("DCR_POOL_GENERIC")) {
    const long long total2 = static_cast<long long>(B) * p.OH * ((p.OW + 1) / 2) * (C / 8);
    maxpool3_bf16_kernel<<<grid_for(total2, 256, di->num_sms), 256, 0, stream>>>(p);
  } else if (!is_max && planes == 1 && k == 3 && !tuning_flag("DCR_POOL_GENERIC")) {
    avgpool3_bf16_kernel<<<grid_for(total, 256, di->num_sms), 256, 0, stream>>>(p);
  } else if (is_max) pool_kernel<true><<<grid_for(total, 256, di->num_sms), 256, 0, stream>>>(p);
  else pool_kernel<false><<<grid_for(total, 256, di->num_sms), 256, 0, stream>>>(p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int reduce_hw(bool gem, const __nv_bfloat16* in, long long in_plane_stride, int planes, int B, int HW, int C,
              float p_exp, float eps, __nv_bfloat16* out, long long out_plane_stride, float* out_f32,
              cudaStream_t stream) {
  DCR_REQUIRE(C % 8 == 0, "reduce_hw: C must be a multiple of 8");
  ReduceHWParams p;
  p.in = in; p.in_plane_stride = in_plane_stride; p.planes = planes; p.B = B; p.HW = HW; p.C = C;
  p.p_exp = p_exp; p.eps = eps; p.out = out; p.out_plane_stride = out_plane_stride; p.out_f32 = out_f32;
  if (B == 0) return 0;
  const int cg = C / 8;
  dim3 grid(B, (cg + 63) / 64);
  if (gem && p_exp == 3.f) reduce_hw_kernel<true, true><<<grid, 64 * kRedSlices, 0, stream>>>(p);
  else if (gem) reduce_hw_kernel<true, false><<<grid, 64 * kRedSlices, 0, stream>>>(p);
  else reduce_hw_kernel<false, false><<<grid, 64 * kRedSlices, 0, stream>>>(p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int layernorm(const __nv_bfloat16* in, long long in_plane_stride, int planes, int rows, int C, long long in_row_stride,
              const float* gamma, const float* beta, float eps, __nv_bfloat16* out, long long out_plane_stride,
              float* out_f32, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(C % 8 == 0 && C <= 1024, "layernorm: C=%d must be a multiple of 8 and <= 1024", C);
  LayerNormParams p;
  p.in = in; p.in_plane_stride = in_plane_stride; p.planes = planes; p.rows = rows; p.C = C;
  p.in_row_stride = in_row_stride; p.gamma = gamma; p.beta = beta; p.eps = eps;
  p.out = out; p.out_plane_stride = out_plane_stride; p.out_f32 = out_f32;
  if (rows == 0) return 0;
  if (planes == 1 && C % 128 == 0 && C / 128 >= 3 && C / 128 <= 8 && in_row_stride % 8 == 0) {
    const int blocks = std::min((rows + 15) / 16, di->num_sms * 8);        // 16 half-warps per 256-thread block
    switch (C / 128) {
      case 3: layernorm_fast_kernel<3><<<blocks, 256, 0, stream>>>(p); break;
      case 4: layernorm_fast_kernel<4><<<blocks, 256, 0, stream>>>(p); break;
      case 6: layernorm_fast_kernel<6><<<blocks, 256, 0, stream>>>(p); break;
      case 8: layernorm_fast_kernel<8><<<blocks, 256, 0, stream>>>(p); break;
      default: layernorm_kernel<<<std::min((rows + 3) / 4, di->num_sms * 32), 128, 0, stream>>>(p); break;
    }
    count_launch();
    DCR_CUDA_CHECK(cudaGetLastError());
    return 0;
  }
  layernorm_kernel<<<std::min((rows + 3) / 4, di->num_sms * 32), 128, 0, stream>>>(p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int vit_tokens(const __nv_bfloat16* patch, long long patch_plane_stride, const float* cls, const float* pos,
               __nv_bfloat16* out, long long out_plane_stride, int planes, int B, int NP, int C, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(C % 8 == 0, "vit_tokens: C must be a multiple of 8");
  VitTokensParams p;
  p.patch = patch; p.patch_plane_stride = patch_plane_stride; p.cls = cls; p.pos = pos; p.out = out;
  p.out_plane_stride = out_plane_stride; p.planes = planes; p.B = B; p.NP = NP; p.C = C;
  if (B == 0) return 0;
  const long long total = static_cast<long long>(B) * (NP + 1) * (C / 8);
  vit_tokens_kernel<<<grid_for(total, 256, di->num_sms), 256, 0, stream>>>(p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace dcr
