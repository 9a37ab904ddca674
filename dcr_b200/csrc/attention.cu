// Multi-head self-attention of the DINO ViT blocks:  softmax(q k^T * scale) v   per (image, head).
// Reference: dino_vits.py:117-128 (Attention.forward): qkv Linear output reshaped to [B, N, 3, heads, dh];
// attn = (q @ k^T) * scale; softmax(dim=-1); x = attn @ v; heads concatenated along the channel dim.
//
// Input  qkv : bf16 planes [B*T, 3*heads*dh] (columns [q | k | v], each heads x dh) -- the fused qkv GEMM output.
// Output out : bf16 planes [B*T, heads*dh].
//
// attention_tc1_kernel (fast mode, one bf16 plane, T <= 256): one CTA per (image, head, 128-row query tile), on tcgen05:
//   S = Q K^T   UMMA 128 x 256 x 16, fp32 in TMEM
//   softmax     4 warps, thread = query row: two passes over the TMEM row (max, then exp2/sum), P written as bf16
//               into a 128B-swizzled K-major shared-memory tile; keys >= T are masked to 0
//   O = P V     UMMA 128 x 64 x 16 with V consumed in place as an MN-major operand (no transpose)
//   epilogue    O / rowsum -> bf16 -> global
// attention_fp32_kernel: exact-fp32 path (parity mode, several planes): K and V of one (image, head) live in shared
// memory as fp32, one warp per query row.  attention_stream_kernel: the same for T > 256.
#include <cuda_bf16.h>

#include "dcr_internal.cuh"
#include "host_util.cuh"
#include "ptx.cuh"

namespace dcr {
namespace {

constexpr uint32_t kFull = 0xffffffffu;

struct AttnParams {
  const __nv_bfloat16* qkv;
  long long qkv_plane_stride;
  __nv_bfloat16* out;
  long long out_plane_stride;
  int planes, B, T, heads, dh;
  float scale;
  int causal;   // 1: query t attends to keys <= t only (CLIP text tower, clip/model.py build_attention_mask)
};

__device__ __forceinline__ float load1(const __nv_bfloat16* base, long long ps, int planes, size_t idx) {
  float v = 0.f;
  for (int p = 0; p < planes; ++p) v += __bfloat162float(base[p * ps + idx]);
  return v;
}

// dh == 64 only (ViT-S/B).  grid = B*heads, block = 256 (8 warps).
__global__ void __launch_bounds__(256) attention_fp32_kernel(const AttnParams p) {
  extern __shared__ __align__(16) float sm[];
  const int T = p.T;
  float* ks = sm;                       // [T][65]
  float* vs = ks + T * 65;              // [T][64]
  float* qs = vs + T * 64;              // [8 warps][64]
  float* ps = qs + 8 * 64;              // [8 warps][Tpad]
  const int Tpad = (T + 31) / 32 * 32;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int ld = 3 * p.heads * 64;
  const size_t row0 = static_cast<size_t>(b) * T;
  for (int i = threadIdx.x; i < T * 64; i += blockDim.x) {
    const int t = i >> 6, d = i & 63;
    ks[t * 65 + d] = load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + t) * ld + p.heads * 64 + h * 64 + d);
    vs[t * 64 + d] = load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + t) * ld + 2 * p.heads * 64 + h * 64 + d);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* q = qs + warp * 64;
  float* pr = ps + warp * Tpad;
  for (int t = warp; t < T; t += 8) {
    q[lane] = load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + t) * ld + h * 64 + lane);
    q[lane + 32] = load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + t) * ld + h * 64 + lane + 32);
    __syncwarp();
    const int TL = p.causal ? t + 1 : T;   // keys this query may see
    float mx = -INFINITY;
    for (int j = lane; j < TL; j += 32) {
      float s = 0.f;
#pragma unroll 16
      for (int d = 0; d < 64; ++d) s = fmaf(q[d], ks[j * 65 + d], s);
      s *= p.scale;
      pr[j] = s;
      mx = fmaxf(mx, s);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, off));
    float sum = 0.f;
    for (int j = lane; j < TL; j += 32) {
      const float e = expf(pr[j] - mx);
      pr[j] = e;
      sum += e;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(kFull, sum, off);
    __syncwarp();
    float o0 = 0.f, o1 = 0.f;
    for (int j = 0; j < TL; ++j) {
      const float w = pr[j];
      o0 = fmaf(w, vs[j * 64 + lane], o0);
      o1 = fmaf(w, vs[j * 64 + lane + 32], o1);
    }
    o0 /= sum;
    o1 /= sum;
    const size_t oidx = (row0 + t) * (p.heads * 64) + h * 64;
    for (int pl = 0; pl < p.planes; ++pl) {
      const __nv_bfloat16 a = __float2bfloat16_rn(o0), c = __float2bfloat16_rn(o1);
      p.out[pl * p.out_plane_stride + oidx + lane] = a;
      p.out[pl * p.out_plane_stride + oidx + lane + 32] = c;
      o0 -= __bfloat162float(a);
      o1 -= __bfloat162float(c);
    }
    __syncwarp();
  }
}

// Long sequences (patch-8 ViTs: 785 tokens, dino_vits.py:381-397): K / V no longer fit in shared memory, so they are
// streamed in tiles of 128 keys and the softmax runs online (running max / sum per query row, output rescaled when the
// max moves).  fp32 SIMT like the kernel above; grid = (B * heads, ceil(T / 64)), one warp owns 8 query rows.
constexpr int kStreamQ = 64;
constexpr int kStreamK = 128;
__global__ void __launch_bounds__(256) attention_stream_kernel(const AttnParams p) {
  extern __shared__ __align__(16) float sm[];
  float* ks = sm;                          // [kStreamK][65]
  float* vs = ks + kStreamK * 65;          // [kStreamK][64]
  float* qs = vs + kStreamK * 64;          // [kStreamQ][64]
  float* ps = qs + kStreamQ * 64;          // [8 warps][kStreamK]
  const int T = p.T;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int q0 = blockIdx.y * kStreamQ;
  const int ld = 3 * p.heads * 64;
  const size_t row0 = static_cast<size_t>(b) * T;
  for (int i = threadIdx.x; i < kStreamQ * 64; i += blockDim.x) {
    const int t = q0 + (i >> 6), d = i & 63;
    qs[i] = t < T ? load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + t) * ld + h * 64 + d) : 0.f;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* pr = ps + warp * kStreamK;
  float m[8], l[8], o0[8], o1[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    m[i] = -INFINITY;
    l[i] = 0.f;
    o0[i] = 0.f;
    o1[i] = 0.f;
  }
  for (int kt = 0; kt < T; kt += kStreamK) {
    __syncthreads();   // previous tile fully consumed (and the query rows staged, first iteration)
    for (int i = threadIdx.x; i < kStreamK * 64; i += blockDim.x) {
      const int j = i >> 6, d = i & 63;
      const bool ok = kt + j < T;
      ks[j * 65 + d] = ok ? load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + kt + j) * ld + p.heads * 64 + h * 64 + d) : 0.f;
      vs[j * 64 + d] = ok ? load1(p.qkv, p.qkv_plane_stride, p.planes, (row0 + kt + j) * ld + 2 * p.heads * 64 + h * 64 + d) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = warp * 8 + i;
      if (q0 + r >= T) continue;   // warp-uniform
      const float* q = qs + r * 64;
      float s[4];
      float tmax = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int j = lane + 32 * c;
        float acc = 0.f;
#pragma unroll 16
        for (int d = 0; d < 64; ++d) acc = fmaf(q[d], ks[j * 65 + d], acc);
        s[c] = (kt + j < T && (!p.causal || kt + j <= q0 + r)) ? acc * p.scale : -INFINITY;
        tmax = fmaxf(tmax, s[c]);
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) tmax = fmaxf(tmax, __shfl_xor_sync(kFull, tmax, off));
      const float m_new = fmaxf(m[i], tmax);          // finite: every tile holds at least one valid key
      const float corr = expf(m[i] - m_new);           // exp(-inf) = 0 on the first tile
      float lsum = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float e = expf(s[c] - m_new);
        pr[lane + 32 * c] = e;
        lsum += e;
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(kFull, lsum, off);
      l[i] = l[i] * corr + lsum;
      __syncwarp();
      float a0 = o0[i] * corr, a1 = o1[i] * corr;
      for (int j = 0; j < kStreamK; ++j) {
        const float w = pr[j];
        a0 = fmaf(w, vs[j * 64 + lane], a0);
        a1 = fmaf(w, vs[j * 64 + lane + 32], a1);
      }
      o0[i] = a0;
      o1[i] = a1;
      m[i] = m_new;
      __syncwarp();
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int t = q0 + warp * 8 + i;
    if (t >= T) continue;
    float a0 = o0[i] / l[i], a1 = o1[i] / l[i];
    const size_t oidx = (row0 + t) * (p.heads * 64) + h * 64;
    for (int pl = 0; pl < p.planes; ++pl) {
      const __nv_bfloat16 x0 = __float2bfloat16_rn(a0), x1 = __float2bfloat16_rn(a1);
      p.out[pl * p.out_plane_stride + oidx + lane] = x0;
      p.out[pl * p.out_plane_stride + oidx + lane + 32] = x1;
      a0 -= __bfloat162float(x0);
      a1 -= __bfloat162float(x1);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// tcgen05 attention
DCR_DEVICE uint64_t umma_desc_sw128_mn(uint32_t smem_addr) {
  // MN-major operand, 128B swizzle: 64 contiguous elements along MN per row, rows = K, 8-row groups 1024 B apart
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;             // LBO (MN repeat) unused: MN extent is one 64-element atom
  d |= static_cast<uint64_t>(1024 >> 4) << 32;     // SBO: next group of 8 K-rows
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

struct AttnTcParams {
  __nv_bfloat16* out;   // [B*T, heads*64]
  int B, T, heads;
  float scale_log2e;    // scale * log2(e)
  int causal;           // 1: keys beyond the query's own position are masked
};

// One query tile per CTA, two CTAs per SM.  A CTA owns ONE 128-row query tile of one (image, head); its P tile
// (128 x 256 bf16 = 64 KB) is written over the Q and K tiles, which are dead once the S MMAs have retired, so a CTA needs
// 96 KB and two of them share an SM (and its 512 TMEM columns, 256 each): one CTA's loads and MMAs run under the other's
// softmax.  K / V of an (image, head) are fetched by both of its CTAs (second fetch: L2).  The earlier form with one CTA
// per (image, head) kept Q (2 tiles), K, V and both P tiles resident (224 KB), so load -> QK^T -> softmax -> PV -> store
// ran as a serial chain on one CTA per SM: 144 us per ViT-S/16 layer at batch 256, ~106 TFLOP/s (removed after commit
// 997ac6f).
constexpr int kAttn1Threads = 160;   // warps 0-3 softmax + epilogue, warp 4 TMA + MMA issue
DCR_DEVICE float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
DCR_DEVICE uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t w;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w) : "f"(hi), "f"(lo));   // upper half <- first source
  return w;
}
// running maximum over one 32-column chunk of a score row; columns >= lim are not part of the row
DCR_DEVICE float chunk_max(const uint32_t (&r)[32], int c0, int lim, float mx) {
  if (c0 + 32 <= lim) {
#pragma unroll
    for (int c = 0; c < 32; c += 2) mx = fmaxf(mx, fmaxf(__uint_as_float(r[c]), __uint_as_float(r[c + 1])));
  } else {
#pragma unroll
    for (int c = 0; c < 32; ++c)
      if (c0 + c < lim) mx = fmaxf(mx, __uint_as_float(r[c]));
  }
  return mx;
}
__global__ void __launch_bounds__(kAttn1Threads, 2)
    attention_tc1_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const AttnTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_q = smem;                 // [128 x 64] bf16          } the P tile (4 k-blocks x [128 x 64]) overwrites
  uint8_t* s_k = s_q + 16384;          // [256 x 64]               } these 64 KB after S = Q K^T
  uint8_t* s_v = s_k + 32768 + 16384;  // [256 x 64] (after 16 KB that only P uses)
  uint8_t* s_p = s_q;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_v + 32768);
  uint64_t* bar_load = bars;
  uint64_t* s_full = bars + 1;
  uint64_t* p_ready = bars + 2;        // 128 arrivals
  uint64_t* o_full = bars + 3;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_mtiles = (p.T + 127) / 128;
  const int mt = blockIdx.x % n_mtiles;
  const int bh = blockIdx.x / n_mtiles;
  const int b = bh / p.heads, h = bh % p.heads;
  const int row0 = b * p.T;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmap_qkv);
    mbar_init(bar_load, 1);
    mbar_init(s_full, 1);
    mbar_init(p_ready, 128);
    mbar_init(o_full, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc<1>(tmem_slot, 256);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    const int cq = h * 64, ck = p.heads * 64 + h * 64, cv = 2 * p.heads * 64 + h * 64;
    if (elect_one()) {
      mbar_arrive_expect_tx(bar_load, 5 * 16384);
      tma_load_2d<1>(s_q, &tmap_qkv, bar_load, cq, row0 + mt * 128, kEvictFirst);
      tma_load_2d<1>(s_k, &tmap_qkv, bar_load, ck, row0, kEvictNormal);
      tma_load_2d<1>(s_k + 16384, &tmap_qkv, bar_load, ck, row0 + 128, kEvictNormal);
      tma_load_2d<1>(s_v, &tmap_qkv, bar_load, cv, row0, kEvictNormal);
      tma_load_2d<1>(s_v + 16384, &tmap_qkv, bar_load, cv, row0 + 128, kEvictNormal);
    }
    __syncwarp();
    mbar_wait(bar_load, 0);
    tc_fence_after();
    constexpr uint32_t idesc_s = umma_idesc_bf16(128, 256);
    constexpr uint32_t idesc_o = umma_idesc_bf16(128, 64) | (1u << 16);   // B operand MN-major
    {
      const uint64_t da = umma_desc_sw128(smem_u32(s_q));
      const uint64_t db = umma_desc_sw128(smem_u32(s_k));
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16<1>(tmem_base, da + 2 * k, db + 2 * k, idesc_s, k != 0);
        umma_commit<1>(s_full);
      }
      __syncwarp();
    }
    mbar_wait(p_ready, 0);
    tc_fence_after();
    if (elect_one()) {
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        const uint64_t da = umma_desc_sw128(smem_u32(s_p + kb * 16384));
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t dv = umma_desc_sw128_mn(smem_u32(s_v + (kb * 64 + k * 16) * 128));
          umma_f16<1>(tmem_base, da + 2 * k, dv, idesc_o, (kb | k) != 0);
        }
      }
      umma_commit<1>(o_full);
    }
    __syncwarp();
  } else {
    const uint32_t quad = warp & 3;
    const uint32_t row = quad * 32 + lane;
    const uint32_t taddr = tmem_base + ((quad * 32u) << 16);
    const uint32_t sw = row & 7;
    mbar_wait(s_full, 0);     // S complete: the MMAs have finished reading Q and K, P may overwrite them
    tc_fence_after();
    const int lim = p.causal ? min(p.T, mt * 128 + static_cast<int>(row) + 1) : p.T;
    // Both passes over the S row are software pipelined: the TMEM load of chunk i+1 is in flight while chunk i is processed
    // (tcgen05.ld is asynchronous until tcgen05.wait::ld; the waits are tied to the registers they guard).
    const int nch = (p.T + 31) / 32;                       // 32-column chunks that hold valid keys (<= 8)
    float mx = -INFINITY;
    {
      uint32_t ra[32], rb[32];
      tmem_ld_32x32(taddr, ra);
#pragma unroll 1
      for (int ch = 0; ch < nch; ch += 2) {
        tmem_ld_wait_regs(ra);
        if (ch + 1 < nch) tmem_ld_32x32(taddr + (ch + 1) * 32, rb);
        mx = chunk_max(ra, ch * 32, lim, mx);
        if (ch + 1 < nch) {
          tmem_ld_wait_regs(rb);
          if (ch + 2 < nch) tmem_ld_32x32(taddr + (ch + 2) * 32, ra);
          mx = chunk_max(rb, (ch + 1) * 32, lim, mx);
        }
      }
    }
    const float mxs = mx * p.scale_log2e;
    float sum = 0.f;
    // exp2, row sum, P chunk -> shared memory.  ~5 instructions per element: FFMA, MUFU.EX2 (approx), half a bf16x2 pack, one
    // shift / mask to get the ROUNDED weight back (the sum must be of the values the tensor core will use) and the add.
    auto emit = [&](int ch, const uint32_t (&r)[32], bool valid) {
      uint32_t pk[16];
      const int c0 = ch * 32;
      if (valid && c0 + 32 <= lim) {               // whole chunk visible: no per-element masks
#pragma unroll
        for (int c = 0; c < 32; c += 2) {
          const float e0 = ex2_approx(fmaf(__uint_as_float(r[c]), p.scale_log2e, -mxs));
          const float e1 = ex2_approx(fmaf(__uint_as_float(r[c + 1]), p.scale_log2e, -mxs));
          const uint32_t w = pack_bf16x2(e0, e1);
          pk[c >> 1] = w;
          sum += __uint_as_float(w << 16) + __uint_as_float(w & 0xffff0000u);
        }
      } else {
#pragma unroll
        for (int c = 0; c < 32; c += 2) {
          const float e0 = (valid && c0 + c < lim) ? ex2_approx(fmaf(__uint_as_float(r[c]), p.scale_log2e, -mxs)) : 0.f;
          const float e1 = (valid && c0 + c + 1 < lim) ? ex2_approx(fmaf(__uint_as_float(r[c + 1]), p.scale_log2e, -mxs)) : 0.f;
          const uint32_t w = pack_bf16x2(e0, e1);
          pk[c >> 1] = w;
          sum += __uint_as_float(w << 16) + __uint_as_float(w & 0xffff0000u);
        }
      }
      uint8_t* prow = s_p + (ch >> 1) * 16384 + row * 128;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(prow + ((((ch & 1) * 4 + j) ^ sw) << 4)) = make_uint4(pk[j * 4], pk[j * 4 + 1], pk[j * 4 + 2], pk[j * 4 + 3]);
    };
    {
      uint32_t ra[32], rb[32];
      tmem_ld_32x32(taddr, ra);
#pragma unroll 1
      for (int ch = 0; ch < 8; ch += 2) {
        const bool va = ch < nch, vb = ch + 1 < nch;
        if (va) tmem_ld_wait_regs(ra);
        if (vb) tmem_ld_32x32(taddr + (ch + 1) * 32, rb);
        emit(ch, ra, va);
        if (vb) tmem_ld_wait_regs(rb);
        if (ch + 2 < nch) tmem_ld_32x32(taddr + (ch + 2) * 32, ra);
        emit(ch + 1, rb, vb);
      }
    }
    fence_proxy_async();     // P (generic proxy) -> visible to the tensor core's async proxy
    tc_fence_before();
    mbar_arrive(p_ready);
    mbar_wait(o_full, 0);
    tc_fence_after();
    const int t = mt * 128 + static_cast<int>(row);
    const float inv = 1.f / sum;
#pragma unroll 1
    for (int ch = 0; ch < 2; ++ch) {
      uint32_t r[32];
      tmem_ld_32x32(taddr + ch * 32, r);
      tmem_ld_wait_regs(r);
      if (t < p.T) {
        __nv_bfloat16* op = p.out + static_cast<size_t>(row0 + t) * (p.heads * 64) + h * 64 + ch * 32;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 v;
          __nv_bfloat162 t0 = __floats2bfloat162_rn(__uint_as_float(r[j * 8 + 0]) * inv, __uint_as_float(r[j * 8 + 1]) * inv);
          __nv_bfloat162 t1 = __floats2bfloat162_rn(__uint_as_float(r[j * 8 + 2]) * inv, __uint_as_float(r[j * 8 + 3]) * inv);
          __nv_bfloat162 t2 = __floats2bfloat162_rn(__uint_as_float(r[j * 8 + 4]) * inv, __uint_as_float(r[j * 8 + 5]) * inv);
          __nv_bfloat162 t3 = __floats2bfloat162_rn(__uint_as_float(r[j * 8 + 6]) * inv, __uint_as_float(r[j * 8 + 7]) * inv);
          v.x = *reinterpret_cast<uint32_t*>(&t0);
          v.y = *reinterpret_cast<uint32_t*>(&t1);
          v.z = *reinterpret_cast<uint32_t*>(&t2);
          v.w = *reinterpret_cast<uint32_t*>(&t3);
          *reinterpret_cast<uint4*>(op + j * 8) = v;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<1>(tmem_base, 256);
}

}  // namespace

int attention(const __nv_bfloat16* qkv, long long qkv_plane_stride, __nv_bfloat16* out, long long out_plane_stride,
              int planes, int B, int T, int heads, int dh, float scale, cudaStream_t stream, int causal) {
  DCR_REQUIRE(dh == 64, "attention: head dim %d not supported (64 only)", dh);
  DCR_REQUIRE(T >= 1 && T <= 16384, "attention: sequence length %d out of range", T);
  if (B == 0) return 0;
  if (planes == 1 && T <= 256) {   // one query tile per CTA, two CTAs per SM
    const DeviceInfo* di = device_info();
    if (!di) return -2;
    CUtensorMap tm;
    if (int rc = make_tmap_2d_bf16(&tm, qkv, static_cast<uint64_t>(B) * T, 3 * heads * 64, 3 * heads * 64, 128, 64)) return rc;
    AttnTcParams tp;
    tp.out = out; tp.B = B; tp.T = T; tp.heads = heads; tp.causal = causal;
    tp.scale_log2e = scale * 1.4426950408889634f;
    const size_t smem1 = 1024 + 16384 + 32768 + 16384 + 32768 + 256;
    DCR_CUDA_CHECK(cudaFuncSetAttribute(attention_tc1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem1)));
    attention_tc1_kernel<<<B * heads * ((T + 127) / 128), kAttn1Threads, smem1, stream>>>(tm, tp);
    count_launch();
    DCR_CUDA_CHECK(cudaGetLastError());
    return 0;
  }
  AttnParams p;
  p.qkv = qkv; p.qkv_plane_stride = qkv_plane_stride; p.out = out; p.out_plane_stride = out_plane_stride;
  p.planes = planes; p.B = B; p.T = T; p.heads = heads; p.dh = dh; p.scale = scale; p.causal = causal;
  if (T > 256) {   // K / V streamed in tiles, online softmax (patch-8 ViTs)
    const size_t smem_s = (static_cast<size_t>(kStreamK) * 65 + kStreamK * 64 + kStreamQ * 64 + 8 * kStreamK) * 4;
    DCR_CUDA_CHECK(cudaFuncSetAttribute(attention_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem_s)));
    attention_stream_kernel<<<dim3(B * heads, (T + kStreamQ - 1) / kStreamQ), 256, smem_s, stream>>>(p);
    count_launch();
    DCR_CUDA_CHECK(cudaGetLastError());
    return 0;
  }
  const int Tpad = (T + 31) / 32 * 32;
  const size_t smem = (static_cast<size_t>(T) * 65 + static_cast<size_t>(T) * 64 + 8 * 64 + 8 * Tpad) * 4;
  DCR_CUDA_CHECK(cudaFuncSetAttribute(attention_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
  attention_fp32_kernel<<<B * heads, 256, smem, stream>>>(p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace dcr
