// Fused all-pairs similarity + per-query top-k for sm_100a.
//
// Replaces (reference = somepago/DCR):
//   diff_retrieval.py:402      sim = torch.mm(values_features, query_features.T)          (fp32, [G,Q], CPU/MKL)
//   diff_retrieval.py:417,613,621   simscores.topk(k, axis=1, largest=True)               k in {1,10}
//   diff_retrieval.py:403,418-419   sim2 = mm(values, values.T); topk(2)[...,-1]           (same kernel, Q:=G, k=2)
//   embedding_search/similarity_search.py:62-63   features @ batch.T ; max(dim=0)
//
// The [Q,G] score matrix is never written.  Three stages, all on the caller's stream:
//   1. to_bf16_rows_kernel   fp32 descriptors -> zero-padded bf16 rows + per-row norms of the rounding residual
//   2. sim_topk_kernel       tcgen05 bf16 GEMM (fp32 accumulate in TMEM) whose epilogue keeps, per query, the
//                            kp (>= k) best approximate scores of its gallery segment (threshold filter on the
//                            accumulator registers, warp-cooperative compaction in shared memory)
//   3. rescore_select_kernel exact re-score (fp64 accumulate, fixed order) of the <= slots*kp candidates per query,
//                            final order (score desc, gallery index asc), plus a per-query certificate that no
//                            non-candidate can reach the k-th exact score.  Queries failing the certificate are
//                            recomputed by brute force in fp64 (exact_scan_kernel / exact_select_kernel).
// Result: indices identical to ranking all G exact dot products with ties broken by lowest index.
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>
#include <type_traits>

#include "dcr_internal.cuh"
#include "host_util.cuh"
#include "ptx.cuh"

namespace dcr {

namespace {

constexpr int kBlockM = 128;      // query rows per CTA (TMEM lanes)
constexpr int kBlockN = 256;      // gallery rows per tile (TMEM columns per accumulator buffer)
constexpr int kBlockK = 64;       // bf16 elements per 128-byte swizzled smem row
constexpr int kMaxKB = 8;         // d_pad <= 512: the query tile stays resident in shared memory; larger: streamed
constexpr int kMaxDim = 8192;     // largest descriptor dimension accepted
constexpr int kKPMax = 32;        // max candidates kept per (query, segment)
constexpr int kWarmTiles = 4;     // tiles replayed at the start of every segment to seed the threshold
constexpr uint32_t kFull = 0xffffffffu;
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KB
constexpr int kMaxSlotsPerQuery = 512;  // (chunk, unit) segments that may cover one q-tile
constexpr int kCG = 2;            // CTAs per work unit: a CTA pair (cta_group::2)

struct SimParams {
  int nq, ng;
  int num_kb;          // d_pad / 64
  int stream_a;        // 1 (d_pad > 512): query k-blocks travel with the gallery k-blocks instead of staying resident
  int n_qtiles;        // ceil(nq / (128*CG))
  int n_gtiles;        // ceil(ng / 256)
  int gchunk;          // gallery tiles per L2-sized chunk (all units sweep chunk c before chunk c+1)
  int n_chunks;
  int kp;              // candidates kept per (query, segment): 8, 16 or 32
  int cap;             // shared-memory list capacity per query row (kp + 16 .. 64)
  int stages;          // B pipeline depth
  uint2* cand;         // [n_slots][rows_per_qtile][kKPMax]   (score bits, local gallery row)
  int* cand_cnt;       // [n_slots][rows_per_qtile]
  float* cand_thr;     // [n_slots][rows_per_qtile]
  const int* bias_flag;    // device flag: 0 = ignore col_bias (query centring switched off for this data)
  const float* col_bias;   // [ng_pad] per-gallery-row score offset nu.(g-mu) added to every accumulator column; null = none
  const float* thr_init;   // per query row: start thresholds (second-chance pass); null = seed by warm-up replay
  unsigned int* gthr;      // [nq_pad] per query row: best threshold any unit has reached so far, as an order-preserving
                           // unsigned key (0 = none); null = no sharing
  unsigned long long* clk; // [4] clock64 / globaltimer at the start and end of CTA 0 (SM clock under this kernel); null = off
};

// ------------------------------------------------------------------------------------------------------------
// stage 1: fp32 rows -> bf16 rows (zero padded to [n_pad, d_pad]) + norms needed by the error bound
//   norms[0][r] = ||bf16(x_r)||, norms[1][r] = ||x_r - bf16(x_r)||, gmax[0] = max_r ||x_r||, gmax[1] = max_r residual
// mu (optional): a vector subtracted from every row before rounding (gallery centring: q.g = q.(g-mu) + q.mu and the
// second term does not depend on g, so the ranking is unchanged while the bf16 rounding error now scales with the
// SPREAD of the gallery instead of its norm).
template <int kIter>
__global__ void __launch_bounds__(256) to_bf16_rows_kernel(const float* __restrict__ x, int n, int d, int n_pad, int d_pad,
                                    const float* __restrict__ mu, __nv_bfloat16* __restrict__ out,
                                    float* __restrict__ norm_hat, float* __restrict__ norm_res,
                                    float* __restrict__ norm_x, unsigned int* __restrict__ gmax,
                                    const float* __restrict__ nu, float* __restrict__ bias_out,
                                    const int* __restrict__ mu_flag, const int* __restrict__ nu_flag) {
  if (mu_flag && *mu_flag == 0) mu = nullptr;   // device-side decision (centre_decision_kernel)
  if (nu_flag && *nu_flag == 0) nu = nullptr;
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  // gmax: one global atomic per BLOCK (100k same-address atomics, one per row, serialise in L2 and dominated this kernel)
  __shared__ unsigned int s_gmax[2];
  if (threadIdx.x < 2) s_gmax[threadIdx.x] = 0u;
  __syncthreads();
  unsigned int w_nx = 0u, w_nr = 0u;   // this warp's running maxima (lane 0)
  for (int row = blockIdx.x * warps_per_block + (threadIdx.x >> 5); row < n_pad; row += gridDim.x * warps_per_block) {
    float s_hat = 0.f, s_res = 0.f, s_x = 0.f;
    double s_bias = 0.0;   // nu . (x - mu) in fp64: the per-gallery-row score offset of query centring
    __nv_bfloat16* o = out + static_cast<size_t>(row) * d_pad;
    if (row < n) {
      const float* xr = x + static_cast<size_t>(row) * d;
      // kIter float4 loads per lane issued back to back (the row's whole HBM read is in flight before the first value
      // is used: the kernel is a pure stream, 12 B/element read+written, and was latency bound with one load at a time)
      for (int c0 = 0; c0 < d_pad; c0 += 128 * kIter) {
        float4 v[kIter];
#pragma unroll
        for (int i = 0; i < kIter; ++i) {
          const int c = c0 + i * 128 + lane * 4;
          v[i] = (c + 3 < d) ? *reinterpret_cast<const float4*>(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);   // d % 4 == 0
        }
#pragma unroll
        for (int i = 0; i < kIter; ++i) {
          const int c = c0 + i * 128 + lane * 4;
          if (c >= d_pad) continue;
          if (c + 3 < d) {
            if (mu) {
              const float4 m = *reinterpret_cast<const float4*>(mu + c);
              v[i].x -= m.x; v[i].y -= m.y; v[i].z -= m.z; v[i].w -= m.w;
            }
            if (nu) {
              const float4 u = *reinterpret_cast<const float4*>(nu + c);
              s_bias = fma(static_cast<double>(u.x), static_cast<double>(v[i].x), s_bias);
              s_bias = fma(static_cast<double>(u.y), static_cast<double>(v[i].y), s_bias);
              s_bias = fma(static_cast<double>(u.z), static_cast<double>(v[i].z), s_bias);
              s_bias = fma(static_cast<double>(u.w), static_cast<double>(v[i].w), s_bias);
            }
          }
          const __nv_bfloat16 h0 = __float2bfloat16_rn(v[i].x), h1 = __float2bfloat16_rn(v[i].y);
          const __nv_bfloat16 h2 = __float2bfloat16_rn(v[i].z), h3 = __float2bfloat16_rn(v[i].w);
          const float f0 = __bfloat162float(h0), f1 = __bfloat162float(h1), f2 = __bfloat162float(h2), f3 = __bfloat162float(h3);
          s_hat += f0 * f0 + f1 * f1 + f2 * f2 + f3 * f3;
          s_res += (v[i].x - f0) * (v[i].x - f0) + (v[i].y - f1) * (v[i].y - f1) + (v[i].z - f2) * (v[i].z - f2) + (v[i].w - f3) * (v[i].w - f3);
          s_x += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
          uint2 pk;
          pk.x = static_cast<uint32_t>(__bfloat16_as_ushort(h0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(h1)) << 16);
          pk.y = static_cast<uint32_t>(__bfloat16_as_ushort(h2)) | (static_cast<uint32_t>(__bfloat16_as_ushort(h3)) << 16);
          *reinterpret_cast<uint2*>(o + c) = pk;
        }
      }
    } else {
      for (int c = lane * 2; c < d_pad; c += 64) *reinterpret_cast<uint32_t*>(o + c) = 0u;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      s_hat += __shfl_xor_sync(kFull, s_hat, off);
      s_res += __shfl_xor_sync(kFull, s_res, off);
      s_x += __shfl_xor_sync(kFull, s_x, off);
      s_bias += __shfl_xor_sync(kFull, s_bias, off);
    }
    if (lane == 0 && bias_out) bias_out[row] = (row < n) ? static_cast<float>(s_bias) : 0.f;
    if (lane == 0 && row < n) {
      // 1.0001: cover the fp32 rounding of the squared sums so the stored values are upper bounds
      float nh = sqrtf(s_hat) * 1.0001f, nr = sqrtf(s_res) * 1.0001f, nx = sqrtf(s_x) * 1.0001f;
      if (norm_hat) norm_hat[row] = nh;
      if (norm_res) norm_res[row] = nr;
      if (norm_x) norm_x[row] = nx;
      w_nx = max(w_nx, __float_as_uint(nx));     // non-negative floats order like their bit patterns
      w_nr = max(w_nr, __float_as_uint(nr));
    }
  }
  if (gmax) {
    if (lane == 0) {
      atomicMax(&s_gmax[0], w_nx);
      atomicMax(&s_gmax[1], w_nr);
    }
    __syncthreads();
    if (threadIdx.x < 2) atomicMax(gmax + threadIdx.x, s_gmax[threadIdx.x]);
  }
}

// column sums of x[n, d] accumulated in double; mean = sum / n afterwards (rows r*row_stride, r < n: any fixed vector works
// as the centre, so a strided sample of the gallery is enough).  A thread owns one 16-byte column group and a slice of the
// block's rows (independent loads, four in flight), the slices meet in shared memory and the block does ONE atomicAdd per
// column: the first version had 592 blocks each add all d columns -- 300k same-address double atomics, 22 us for a 16 MB sample.
constexpr int kColSumThreads = 512;
__global__ void __launch_bounds__(kColSumThreads)
    col_sum_kernel(const float* __restrict__ x, int n, int row_stride, int d, double* __restrict__ sums,
                   double* __restrict__ sq_sums) {
  __shared__ double red[kColSumThreads][8];
  const int groups = d >> 2;                                   // d % 4 == 0 (checked by the caller)
  const int G = min(groups, kColSumThreads), S = kColSumThreads / G;
  const int tg = threadIdx.x % G, sl = threadIdx.x / G;         // threads with sl >= S idle (G does not divide the block)
  const int rows_per_block = (n + gridDim.x - 1) / gridDim.x;
  const int r0 = blockIdx.x * rows_per_block, r1 = min(n, r0 + rows_per_block);
  for (int cg = tg; cg < groups; cg += G) {
    double da[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) da[e] = 0.0;
    if (sl < S) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
      int cnt = 0;
#pragma unroll 4
      for (int r = r0 + sl; r < r1; r += S) {
        const float4 v = *reinterpret_cast<const float4*>(x + static_cast<size_t>(r) * row_stride * d + cg * 4);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        acc2.x += v.x * v.x; acc2.y += v.y * v.y; acc2.z += v.z * v.z; acc2.w += v.w * v.w;
        if (++cnt == 256) {   // flush the fp32 partials into the double accumulators every 256 rows
          da[0] += acc.x; da[1] += acc.y; da[2] += acc.z; da[3] += acc.w;
          da[4] += acc2.x; da[5] += acc2.y; da[6] += acc2.z; da[7] += acc2.w;
          acc = make_float4(0.f, 0.f, 0.f, 0.f);
          acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
          cnt = 0;
        }
      }
      da[0] += acc.x; da[1] += acc.y; da[2] += acc.z; da[3] += acc.w;
      da[4] += acc2.x; da[5] += acc2.y; da[6] += acc2.z; da[7] += acc2.w;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) red[threadIdx.x][e] = da[e];
    __syncthreads();
    if (sl == 0 && r1 > r0) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        double t = 0.0;
        for (int s2 = 0; s2 < S; ++s2) t += red[s2 * G + tg][e];   // fixed order within the block
        if (e < 4) atomicAdd(sums + cg * 4 + e, t);
        else if (sq_sums) atomicAdd(sq_sums + cg * 4 + (e - 4), t);
      }
    }
    __syncthreads();
  }
}
__global__ void col_mean_finish_kernel(const double* __restrict__ sums, int n, int d, float* __restrict__ mu) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < d) mu[c] = static_cast<float>(sums[c] / n);
}
// Query centring pays only when the centred queries are much shorter than the queries themselves (the bf16 error
// bound shrinks by ||q-nu|| / ||q||) -- and costs a per-column offset in the fused epilogue.  flag = 1 when the
// mean squared norm of the centred sample is below 1/16 of the uncentred one (a 4x tighter bound).
__global__ void __launch_bounds__(256)
    centre_decision_kernel(const double* __restrict__ sums, const double* __restrict__ sq_sums, int n, int d,
                           int* __restrict__ flag) {
  __shared__ double s_m2[8], s_nu2[8];
  double m2 = 0.0, nu2 = 0.0;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    m2 += sq_sums[c] / n;
    const double m = sums[c] / n;
    nu2 += m * m;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    m2 += __shfl_xor_sync(kFull, m2, off);
    nu2 += __shfl_xor_sync(kFull, nu2, off);
  }
  if ((threadIdx.x & 31) == 0) {
    s_m2[threadIdx.x >> 5] = m2;
    s_nu2[threadIdx.x >> 5] = nu2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    m2 = nu2 = 0.0;
    for (int w = 0; w < 8; ++w) {
      m2 += s_m2[w];
      nu2 += s_nu2[w];
    }
    *flag = (m2 - nu2 < m2 / 16.0) ? 1 : 0;
  }
}

// second-chance pass: copy the bf16 rows of the flagged queries into a compact matrix (zero rows up to n_pad)
__global__ void gather_rows_kernel(const __nv_bfloat16* __restrict__ src, const int* __restrict__ rows, int n, int n_pad,
                                   int d_pad, __nv_bfloat16* __restrict__ dst) {
  const int chunks = d_pad / 8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
       i < static_cast<long long>(n_pad) * chunks; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / chunks), c = static_cast<int>(i % chunks);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < n) v = *reinterpret_cast<const uint4*>(src + static_cast<size_t>(rows[r]) * d_pad + c * 8);
    *reinterpret_cast<uint4*>(dst + static_cast<size_t>(r) * d_pad + c * 8) = v;
  }
}

// ------------------------------------------------------------------------------------------------------------
// stage 2 helpers

DCR_DEVICE unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// order-preserving float <-> unsigned key (0 is below every float): thresholds are shared with atomicMax
DCR_DEVICE unsigned int thr_key(float f) {
  const unsigned int b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
DCR_DEVICE float thr_from_key(unsigned int k) {
  if (k == 0) return -INFINITY;
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

DCR_DEVICE float max8(const float* v) {
  return fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), fmaxf(fmaxf(v[4], v[5]), fmaxf(v[6], v[7])));
}

DCR_DEVICE void tmem_ld_wait_dep(uint32_t (&r)[32]) {
  // the registers are tied to the wait so that no consumer of r[] can be scheduled above it
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                 "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                 "+r"(r[29]), "+r"(r[30]), "+r"(r[31])::"memory");
}

// Keep the kp best of lane L's n (kp < n <= 64) list entries, stored at list[j * 128] (j = 0..n-1); returns the
// kp-th best score, which becomes that row's new threshold.  Whole warp cooperates: lane l ranks entries l and
// l+32 against all n keys (broadcast shared-memory reads), winners are rewritten in rank order (sorted list).
DCR_DEVICE float compact_one(uint2* list, int n, int kp, uint32_t lane) {
  const uint2 none = make_uint2(0xff800000u, 0xffffffffu);  // -inf
  const int l0 = static_cast<int>(lane), l1 = l0 + 32;
  const uint2 e0 = (l0 < n) ? list[l0 * 128] : none;
  const uint2 e1 = (l1 < n) ? list[l1 * 128] : none;
  const float k0 = __uint_as_float(e0.x), k1 = __uint_as_float(e1.x);
  int r0 = 0, r1 = 0;
  const float* keys = reinterpret_cast<const float*>(list);   // key j at keys[j * 256]
  if (n <= 32) {
#pragma unroll 4
    for (int j = 0; j < n; ++j) {
      const float kj = keys[j * 256];
      r0 += (kj > k0) || (kj == k0 && j < l0);
    }
  } else {
#pragma unroll 4
    for (int j = 0; j < n; ++j) {
      const float kj = keys[j * 256];
      r0 += (kj > k0) || (kj == k0 && j < l0);
      r1 += (kj > k1) || (kj == k1 && j < l1);
    }
  }
  __syncwarp();
  if (l0 < n && r0 < kp) list[r0 * 128] = e0;
  if (l1 < n && r1 < kp) list[r1 * 128] = e1;
  __syncwarp();
  return keys[(kp - 1) * 256];
}

DCR_DEVICE void compact_warp(uint2* warp_list, unsigned need, int kp, float& thr, int& cnt, uint32_t lane) {
  __syncwarp();   // make every lane's list stores visible to the lanes that will rank them
  while (need) {
    const int L = __ffs(need) - 1;
    need &= need - 1;
    const int n = __shfl_sync(kFull, cnt, L);
    const float t = compact_one(warp_list + L, n, kp, lane);
    if (static_cast<int>(lane) == L) {
      thr = t;
      cnt = kp;
    }
  }
}

DCR_DEVICE void st_shared_v2_if(uint32_t saddr, uint32_t a, uint32_t b, bool p) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %3, 0;\n\t"
      "@q st.shared.v2.b32 [%0], {%1, %2};\n\t}\n" ::"r"(saddr),
      "r"(a), "r"(b), "r"(static_cast<uint32_t>(p))
      : "memory");
}

// One 32-column chunk of the accumulator row held by this thread.  The common case (no lane of the warp has a
// score above its threshold) costs a max-tree, one compare and one vote.  Otherwise the 8-column sub-chunks that
// contain a hit are appended to the row lists with predicated stores (no per-lane branching).
template <bool kMaskTail>
DCR_DEVICE void scan_chunk(const uint32_t (&r)[32], const float* sb, int gcol0, int ng, float& thr, int& cnt,
                           uint32_t my_list_saddr, uint2* warp_list, int kp, int cap, uint32_t lane) {
  float v[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) v[c] = __uint_as_float(r[c]);
  if (sb) {   // warp-uniform
#pragma unroll
    for (int c = 0; c < 32; c += 4) {
      const float4 b = *reinterpret_cast<const float4*>(sb + c);
      v[c] += b.x; v[c + 1] += b.y; v[c + 2] += b.z; v[c + 3] += b.w;
    }
  }
#pragma unroll
  for (int c = 0; c < 32; ++c)
    if (kMaskTail && gcol0 + c >= ng) v[c] = -INFINITY;
  float s[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) s[i] = max8(v + 8 * i);
  const float m = fmaxf(fmaxf(s[0], s[1]), fmaxf(s[2], s[3]));
  if (__any_sync(kFull, m > thr)) {
#pragma unroll
    for (int sub = 0; sub < 4; ++sub) {
      if (__any_sync(kFull, s[sub] > thr)) {
        uint32_t addr = my_list_saddr + static_cast<uint32_t>(cnt) * 1024u;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float x = v[sub * 8 + c];
          const bool h = x > thr;
          st_shared_v2_if(addr, __float_as_uint(x), static_cast<uint32_t>(gcol0 + sub * 8 + c), h);
          addr += h ? 1024u : 0u;
        }
        cnt = static_cast<int>((addr - my_list_saddr) >> 10);
        const unsigned need = __ballot_sync(kFull, cnt > cap - 8);
        if (need) compact_warp(warp_list, need, kp, thr, cnt, lane);
      }
    }
  }
}

// last gallery tile only: columns past the end of the gallery never win (-inf survives the offset add)
DCR_DEVICE void mask_tail(uint32_t (&r)[32], int gcol0, int ng) {
#pragma unroll
  for (int c = 0; c < 32; ++c)
    if (gcol0 + c >= ng) r[c] = 0xff800000u;
}

// Warm-up chunk: running maxima of 32 column slots (slot = column mod 32); no candidates are recorded.
template <bool kMaskTail>
DCR_DEVICE void warm_chunk(const uint32_t (&r)[32], const float* sb, int gcol0, int ng, float (&slot)[32]) {
#pragma unroll
  for (int c = 0; c < 32; ++c) {
    float x = __uint_as_float(r[c]);
    if (sb) x += sb[c];
    if (kMaskTail && gcol0 + c >= ng) x = -INFINITY;
    slot[c] = fmaxf(slot[c], x);
  }
}

// Seed of a segment's threshold from the warm-up maxima: fold the 32 slot maxima into `groups` >= kp disjoint groups;
// the smallest group maximum is exceeded by at least groups-1 already-seen scores, so it is a safe (never too high
// for kp) start.  Segments shorter than the warm-up still get a valid bound.
DCR_DEVICE float seed_threshold(float (&slot)[32], int kp) {
  int groups = 32;
  if (kp <= 16) {
#pragma unroll
    for (int c = 0; c < 16; ++c) slot[c] = fmaxf(slot[c], slot[c + 16]);
    groups = 16;
  }
  if (kp <= 8) {
#pragma unroll
    for (int c = 0; c < 8; ++c) slot[c] = fmaxf(slot[c], slot[c + 8]);
    groups = 8;
  }
  if (kp <= 4) {
#pragma unroll
    for (int c = 0; c < 4; ++c) slot[c] = fmaxf(slot[c], slot[c + 4]);
    groups = 4;
  }
  float lo = slot[0];
#pragma unroll
  for (int c = 1; c < 32; ++c)
    if (c < groups) lo = fminf(lo, slot[c]);
  // strictly below the smallest group maximum so that the maxima themselves are recorded
  float thr = (lo == -INFINITY) ? -INFINITY : __uint_as_float(__float_as_uint(lo) + (lo > 0.f ? -1 : (lo < 0.f ? 1 : 0)));
  if (lo == 0.f) thr = -1e-30f;
  return thr;
}

// Work decomposition shared by the three warp roles (and mirrored by rescore_select_kernel): for every gallery chunk
// c (chunks are L2-sized so that the units, which all sweep chunk c at about the same time, share its tiles in L2)
// the (q-tile, g-tile-in-chunk) grid is linearised q-major and cut into n_units equal contiguous ranges; a unit's range
// is walked as segments = maximal runs inside one q-tile.  Thresholds carry over from chunk to chunk: `carried` says
// that this unit finished a segment of the same q-tile before (its final per-row thresholds are valid lower bounds, so
// no warm-up replay is needed).
struct SegWalker {
  int n_qtiles, n_gtiles, gchunk, n_chunks;
  long long unit, n_units;
  // current segment
  int chunk, qi, g_begin, ntiles, slot;
  bool carried;
  // state
  long long t, t_end;
  int ncg, g_lo;
  int tag[4];
  __device__ SegWalker(int nq_t, int ng_t, int gc, int nc, long long u, long long nu)
      : n_qtiles(nq_t), n_gtiles(ng_t), gchunk(gc), n_chunks(nc), unit(u), n_units(nu), chunk(-1), t(0), t_end(0) {
    tag[0] = tag[1] = tag[2] = tag[3] = -1;
  }
  __device__ bool next() {
    if (chunk >= 0) {   // close the previous segment
      const int s4 = qi & 3;
      if (s4 == 0) tag[0] = qi; else if (s4 == 1) tag[1] = qi; else if (s4 == 2) tag[2] = qi; else tag[3] = qi;
    }
    while (t >= t_end) {
      ++chunk;
      if (chunk >= n_chunks) return false;
      g_lo = chunk * gchunk;
      ncg = min(gchunk, n_gtiles - g_lo);
      const long long T = static_cast<long long>(n_qtiles) * ncg;
      t = unit * T / n_units;
      t_end = (unit + 1) * T / n_units;
    }
    qi = static_cast<int>(t / ncg);
    g_begin = g_lo + static_cast<int>(t % ncg);
    const long long seg_end = min(t_end, static_cast<long long>(qi + 1) * ncg);
    ntiles = static_cast<int>(seg_end - t);
    slot = chunk * (static_cast<int>(n_units) + n_qtiles) + static_cast<int>(unit) + qi;
    const int s4 = qi & 3;
    const int tg = s4 == 0 ? tag[0] : (s4 == 1 ? tag[1] : (s4 == 2 ? tag[2] : tag[3]));
    carried = (tg == qi);
    t = seg_end;
    return true;
  }
};

// ------------------------------------------------------------------------------------------------------------
// stage 2: the fused kernel.  A CTA pair per work unit (UMMA 256x256x16, cta_group::2): each CTA keeps its own 128
// queries resident and loads half of every gallery tile, so L2->SMEM traffic per FLOP is half that of one CTA per unit.
//
// Work decomposition: the (q-tile, g-tile) grid is linearised q-major into T = n_qtiles * n_gtiles tiles and cut
// into gridDim/kCG equal contiguous ranges.  A unit's range is walked as "segments" (maximal runs inside one
// q-tile); per segment the query tile is loaded once (A stays resident) and the thresholds are seeded by
// replaying the first kWarmTiles tiles.  Segment (unit u, q-tile i) owns candidate slot u + i.
// kBias: compiled with / without the per-column offset path of query centring.  Both variants are launched; the one
// that does not match the device-side decision (p.bias_flag) exits at once -- no host synchronisation needed.
template <bool kBias, int kSets>
__global__ void __launch_bounds__(64 + 128 * kSets, 1)
    sim_topk_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_g,
                    const SimParams p) {
  if (((p.col_bias != nullptr) && (p.bias_flag != nullptr) && (*p.bias_flag != 0)) != kBias) return;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve-up (all tile bases 1024-byte aligned for the 128B swizzle)
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kBRows = kBlockN / kCG;
  constexpr int kBTileBytes = kBRows * kBlockK * 2;
  // resident mode: [num_kb x 16 KB query tile][stages x gallery tile]; streamed mode (d_pad > 512, the query tile no
  // longer fits): [stages x (gallery tile | 16 KB query k-block)] -- twice the L2->SMEM traffic per FLOP
  const bool stream_a = p.stream_a != 0;
  const int stage_bytes = kBTileBytes + (stream_a ? kATileBytes : 0);
  uint8_t* smem_a = smem;                                                  // num_kb x 16 KB (resident mode)
  uint8_t* smem_b = smem_a + (stream_a ? 0 : p.num_kb * kATileBytes);      // stages x stage_bytes
  uint2* cand = reinterpret_cast<uint2*>(smem_b + p.stages * stage_bytes);  // [kSets][cap][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(cand) + kSets * p.cap * 128 * 8);
  uint64_t* b_full = bars;              // [stages]
  uint64_t* b_empty = bars + 8;         // [stages]
  uint64_t* a_full = bars + 16;
  uint64_t* a_empty = bars + 17;
  uint64_t* t_full = bars + 18;         // [2]
  uint64_t* t_empty = bars + 20;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);
  float* carry = reinterpret_cast<float*>(bars + 32);   // [kSets][4][128] thresholds carried to the next chunk, by q-tile & 3

  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = (cta_rank == 0);

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_g);
  }
  if (warp == 1 && elect_one()) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&b_full[s], kCG);
      mbar_init(&b_empty[s], 1);
    }
    mbar_init(a_full, kCG);
    mbar_init(a_empty, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&t_full[b], 1);
      mbar_init(&t_empty[b], 4 * kSets * kCG);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<kCG>(tmem_slot, 512);
    tmem_relinquish<kCG>();
  }
  tc_fence_before();
  __syncthreads();   // CTA-local ordering of the set-up writes (mbarrier init, TMEM slot) for this CTA's own readers ...
  cluster_sync();   // ... and the peer CTA's barriers are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (p.clk && blockIdx.x == 0 && threadIdx.x == 0) {
    p.clk[0] = clock64();
    p.clk[1] = global_timer_ns();
  }

  // this unit's tile range
  const long long n_units = gridDim.x / kCG;
  const long long unit = blockIdx.x / kCG;
  const int rows_per_qtile = kBlockM * kCG;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    // The whole warp walks the loop (warp-uniform values stay in uniform registers) and one elected lane issues: under
    // `if (lane == 0)` every UTMALDG / UTCHMMA gets an ELECT + R2UR + BRA.U.ANY wrapper, and the single-thread
    // instruction stream is the critical path of the pipeline (tools/microbench/umma_rate.cu).
    {
      uint32_t seg = 0;
      PipeState st(p.stages);
      SegWalker w(p.n_qtiles, p.n_gtiles, p.gchunk, p.n_chunks, unit, n_units);
      while (w.next()) {
        const int qi = w.qi, g_begin = w.g_begin, ntiles = w.ntiles;
        const int warm = (p.thr_init || w.carried) ? 0 : min(kWarmTiles, ntiles);
        const int q_row = qi * rows_per_qtile + static_cast<int>(cta_rank) * kBlockM;
        if (!stream_a) {   // resident query tile
          mbar_wait(a_empty, (seg & 1) ^ 1);
          if (elect_one()) {
            if (leader) mbar_arrive_expect_tx(a_full, p.num_kb * kATileBytes * kCG);
            else mbar_arrive_cluster(a_full, 0);
            for (int kb = 0; kb < p.num_kb; ++kb)
              tma_load_2d<kCG>(smem_a + kb * kATileBytes, &tmap_q, a_full, kb * kBlockK, q_row, kEvictNormal);
          }
          __syncwarp();
        }
        for (int j = 0; j < warm + ntiles; ++j) {
          const int gi = g_begin + (j < warm ? j : j - warm);
          const int g_row = gi * kBlockN + static_cast<int>(cta_rank) * kBRows;
          for (int kb = 0; kb < p.num_kb; ++kb, st.next()) {
            const uint32_t s = st.s, ph = st.ph;
            mbar_wait(&b_empty[s], ph ^ 1);
            if (elect_one()) {
              if (leader) mbar_arrive_expect_tx(&b_full[s], stage_bytes * kCG);
              else mbar_arrive_cluster(&b_full[s], 0);
              tma_load_2d<kCG>(smem_b + s * stage_bytes, &tmap_g, &b_full[s], kb * kBlockK, g_row, kEvictNormal);
              if (stream_a)
                tma_load_2d<kCG>(smem_b + s * stage_bytes + kBTileBytes, &tmap_q, &b_full[s], kb * kBlockK, q_row, kEvictNormal);
            }
            __syncwarp();
          }
        }
        ++seg;
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer (leader CTA) =====================================
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(kBlockM * kCG, kBlockN);
      uint32_t seg = 0, tc = 0;
      PipeState st(p.stages);
      const uint64_t da0 = umma_desc_sw128(smem_u32(stream_a ? smem_b + kBTileBytes : smem_a));
      const uint64_t db0 = umma_desc_sw128(smem_u32(smem_b));
      const uint32_t stage_step = static_cast<uint32_t>(stage_bytes) >> 4;   // descriptor start-address units (16 B)
      SegWalker w(p.n_qtiles, p.n_gtiles, p.gchunk, p.n_chunks, unit, n_units);
      while (w.next()) {
        const int ntiles = w.ntiles;
        const int warm = (p.thr_init || w.carried) ? 0 : min(kWarmTiles, ntiles);
        if (!stream_a) {
          mbar_wait(a_full, seg & 1);
          tc_fence_after();
        }
        for (int j = 0; j < warm + ntiles; ++j, ++tc) {
          const uint32_t buf = tc & 1;
          mbar_wait(&t_empty[buf], ((tc >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + buf * kBlockN;
          for (int kb = 0; kb < p.num_kb; ++kb, st.next()) {
            const uint32_t s = st.s;
            mbar_wait(&b_full[s], st.ph);
            tc_fence_after();
            const uint64_t da = da0 + static_cast<uint64_t>(stream_a ? s * stage_step : static_cast<uint32_t>(kb) * (kATileBytes >> 4));
            const uint64_t db = db0 + static_cast<uint64_t>(s * stage_step);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k)
                umma_f16<kCG>(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);  // +32 B per K=16 step
              umma_commit<kCG>(&b_empty[s]);   // frees this B stage (both CTAs) once the MMAs above retire
              if (kb == p.num_kb - 1) {
                umma_commit<kCG>(&t_full[buf]);
                if (!stream_a && j == warm + ntiles - 1) umma_commit<kCG>(a_empty);
              }
            }
            __syncwarp();
          }
        }
        ++seg;
      }
    }
  } else {
    // ===================================== epilogue warps =====================================
    // kSets = 2: two warps per TMEM lane quadrant, each owning one column half ("set") of every accumulator tile and
    // its own candidate lists / slot -- the filter is issue- and latency-bound with a single warp per sub-partition.
    const uint32_t quad = warp & 3;             // TMEM lane quadrant this warp may read
    const uint32_t set = (warp - 2) >> 2;       // column range [set * kSetCols, (set + 1) * kSetCols) of every tile
    const uint32_t row = quad * 32 + lane;      // query row inside this CTA's tile
    constexpr int kSetCols = kBlockN / kSets;
    uint2* set_list = cand + set * p.cap * 128;
    const uint32_t my_list = smem_u32(set_list + row);
    uint2* warp_list = set_list + quad * 32;
    const uint32_t tmem_row = tmem_base + ((quad * 32u) << 16);
    float* my_carry = carry + set * 4 * kBlockM;
    const int kp = p.kp, cap = p.cap;
    const float* colbias = kBias ? p.col_bias : nullptr;
    uint32_t tc = 0;
    SegWalker w(p.n_qtiles, p.n_gtiles, p.gchunk, p.n_chunks, unit, n_units);
    while (w.next()) {
      const int qi = w.qi, g_begin = w.g_begin, ntiles = w.ntiles;
      const int warm = (p.thr_init || w.carried) ? 0 : min(kWarmTiles, ntiles);
      float thr = -INFINITY;
      if (p.thr_init) {
        const int qrow_g = qi * rows_per_qtile + static_cast<int>(cta_rank) * kBlockM + static_cast<int>(row);
        thr = qrow_g < p.nq ? p.thr_init[qrow_g] : INFINITY;   // padding rows collect nothing
      }
      // a threshold this row reached on an earlier gallery chunk is a valid (and usually tight) start here
      if (w.carried) thr = fmaxf(thr, my_carry[(qi & 3) * kBlockM + row]);
      int cnt = 0;
      // Threshold sharing: a threshold ANY unit reached for this query row (kp recorded scores above it exist somewhere
      // in the gallery) is a valid drop bound for every other unit sweeping the same query tile.  Read once per tile
      // (the load is issued before the accumulator-ready wait), published when it has risen.
      const int qrow_s = qi * rows_per_qtile + static_cast<int>(cta_rank) * kBlockM + static_cast<int>(row);
      unsigned int* gslot = (p.gthr && qrow_s < p.nq) ? p.gthr + qrow_s : nullptr;
      float published = gslot ? thr_from_key(*reinterpret_cast<volatile unsigned int*>(gslot)) : INFINITY;
      if (gslot) thr = fmaxf(thr, published);

      // one accumulator tile: warm-up tiles only track column-slot maxima, the others feed the candidate lists.  Two
      // separate loops so that the 32 slot registers are dead while the lists are live.
      auto tile = [&](auto warm_tag, int gi, float (&slot)[32]) {
        constexpr bool kWarm = decltype(warm_tag)::value;
        const int gcol0 = gi * kBlockN + static_cast<int>(set) * kSetCols;
        const bool tail = gcol0 + kSetCols > p.ng;
        const uint32_t buf = tc & 1;
        const float* sb = kBias ? colbias + gcol0 : nullptr;   // per-column offsets: warp-uniform (broadcast) loads
        unsigned int shared_key = 0;
        if (!kWarm && gslot) shared_key = *reinterpret_cast<volatile unsigned int*>(gslot);
        mbar_wait(&t_full[buf], (tc >> 1) & 1);
        tc_fence_after();
        if (!kWarm && gslot) {
          if (thr > published) {   // risen since the last publication (compaction): let the other units know
            atomicMax(gslot, thr_key(thr));
            published = thr;
          }
          const float other = thr_from_key(shared_key);
          if (other > thr) {
            thr = other;
            published = other;
          }
        }
        const uint32_t taddr = tmem_row + buf * kBlockN + set * kSetCols;
        uint32_t ra[32], rb[32];
        auto release = [&]() {   // this warp's columns of the accumulator buffer are in registers
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&t_empty[buf], 0);
        };
        // TMEM read pipeline: chunk i+1 is in flight while chunk i is scanned
        tmem_ld_32x32(taddr, ra);
#pragma unroll 1
        for (int ch = 0; ch < kSetCols / 32; ch += 2) {
          tmem_ld_wait_dep(ra);
          tmem_ld_32x32(taddr + (ch + 1) * 32, rb);
          if (tail) mask_tail(ra, gcol0 + ch * 32, p.ng);
          if constexpr (kWarm) warm_chunk<false>(ra, sb ? sb + ch * 32 : nullptr, gcol0 + ch * 32, p.ng, slot);
          else scan_chunk<false>(ra, sb ? sb + ch * 32 : nullptr, gcol0 + ch * 32, p.ng, thr, cnt, my_list, warp_list, kp, cap, lane);
          tmem_ld_wait_dep(rb);
          if (ch + 2 < kSetCols / 32) tmem_ld_32x32(taddr + (ch + 2) * 32, ra);
          else release();
          if (tail) mask_tail(rb, gcol0 + (ch + 1) * 32, p.ng);
          if constexpr (kWarm) warm_chunk<false>(rb, sb ? sb + (ch + 1) * 32 : nullptr, gcol0 + (ch + 1) * 32, p.ng, slot);
          else scan_chunk<false>(rb, sb ? sb + (ch + 1) * 32 : nullptr, gcol0 + (ch + 1) * 32, p.ng, thr, cnt, my_list, warp_list, kp, cap, lane);
        }
      };
      if (warm > 0) {
        float slot[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) slot[c] = -INFINITY;
#pragma unroll 1
        for (int j = 0; j < warm; ++j, ++tc) tile(std::true_type{}, g_begin + j, slot);
        thr = seed_threshold(slot, kp);
      }
      {
        float unused[32];
#pragma unroll 1
        for (int j = 0; j < ntiles; ++j, ++tc) tile(std::false_type{}, g_begin + j, unused);
      }
      // ---- flush this segment's lists: final compaction to kp, then coalesced copy to the slot ----
      __syncwarp();
      {
        const unsigned need = __ballot_sync(kFull, cnt > kp);
        if (need) compact_warp(warp_list, need, kp, thr, cnt, lane);
      }
      __syncwarp();
      my_carry[(qi & 3) * kBlockM + row] = thr;
      if (gslot && thr > published) atomicMax(gslot, thr_key(thr));
      const size_t slot_row0 = (static_cast<size_t>(w.slot) * kSets + set) * rows_per_qtile + cta_rank * kBlockM + quad * 32;
      for (int L = 0; L < 32; ++L) {
        const int n = __shfl_sync(kFull, cnt, L);
        if (static_cast<int>(lane) < n) p.cand[(slot_row0 + L) * kKPMax + lane] = warp_list[L + lane * 128];
      }
      p.cand_cnt[slot_row0 + lane] = cnt;
      p.cand_thr[slot_row0 + lane] = thr;
      __syncwarp();
    }
  }

  // teardown
  tc_fence_before();
  cluster_sync();
  if (warp == 2) tmem_dealloc<kCG>(tmem_base, 512);
  if (p.clk && blockIdx.x == 0 && threadIdx.x == 0) {
    p.clk[2] = clock64();
    p.clk[3] = global_timer_ns();
  }
}

// ------------------------------------------------------------------------------------------------------------
// exact dot product, fp64 accumulate, fixed association: lane l owns elements l*4 + 128*i (float4 granules),
// accumulates them in order, then a fixed xor-butterfly.  Used by both the re-score and the brute-force path so
// that the two produce bit-identical values.
DCR_DEVICE double exact_dot_warp(const float* __restrict__ a_smem, const float* __restrict__ b, int d, uint32_t lane) {
  double acc = 0.0;
  for (int c = lane * 4; c < d; c += 128) {
    if (c + 3 < d) {
      const float4 bv = *reinterpret_cast<const float4*>(b + c);
      acc = fma(static_cast<double>(a_smem[c]), static_cast<double>(bv.x), acc);
      acc = fma(static_cast<double>(a_smem[c + 1]), static_cast<double>(bv.y), acc);
      acc = fma(static_cast<double>(a_smem[c + 2]), static_cast<double>(bv.z), acc);
      acc = fma(static_cast<double>(a_smem[c + 3]), static_cast<double>(bv.w), acc);
    } else {
      for (int e = c; e < d; ++e) acc = fma(static_cast<double>(a_smem[e]), static_cast<double>(b[e]), acc);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(kFull, acc, off);
  return acc;
}

// Same values, same association as exact_dot_warp with the query row already widened to fp64 in shared memory (the widening
// is exact): the re-score kernel is bound by the fp64 pipe -- per gallery row 512 fma plus 1024 fp32->fp64 conversions --
// and this halves the conversions.
DCR_DEVICE double exact_dot_warp_qd(const double* __restrict__ a_smem, const float* __restrict__ b, int d, uint32_t lane) {
  double acc = 0.0;
  for (int c = lane * 4; c < d; c += 128) {
    if (c + 3 < d) {
      const float4 bv = *reinterpret_cast<const float4*>(b + c);
      const double2 a01 = *reinterpret_cast<const double2*>(a_smem + c);
      const double2 a23 = *reinterpret_cast<const double2*>(a_smem + c + 2);
      acc = fma(a01.x, static_cast<double>(bv.x), acc);
      acc = fma(a01.y, static_cast<double>(bv.y), acc);
      acc = fma(a23.x, static_cast<double>(bv.z), acc);
      acc = fma(a23.y, static_cast<double>(bv.w), acc);
    } else {
      for (int e = c; e < d; ++e) acc = fma(a_smem[e], static_cast<double>(b[e]), acc);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(kFull, acc, off);
  return acc;
}

// owner unit of linear tile t  (units own [u*T/U, (u+1)*T/U) )
DCR_DEVICE long long owner_unit(long long t, long long T, long long U) { return ((t + 1) * U + T - 1) / T - 1; }

// block-wide arg-best over (score desc, index asc); entries with taken[i] != 0 are skipped
struct Best {
  double s;
  long long i;
  int pos;
};
DCR_DEVICE bool better(double s, long long i, double bs, long long bi) { return (s > bs) || (s == bs && i < bi); }

// block-wide arg-best over (key desc, index asc) of 128 threads; every thread passes its local best (pos < 0 = none)
struct BlockBest {
  double key[4];
  long long idx[4];
  int pos[4];
};
DCR_DEVICE void block_argbest(double& bs, long long& bi, int& bp, BlockBest* sb, uint32_t lane, uint32_t warp) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double os = __shfl_xor_sync(kFull, bs, off);
    const long long oi = __shfl_xor_sync(kFull, bi, off);
    const int op = __shfl_xor_sync(kFull, bp, off);
    if (op >= 0 && (bp < 0 || better(os, oi, bs, bi))) {
      bs = os;
      bi = oi;
      bp = op;
    }
  }
  if (lane == 0) {
    sb->key[warp] = bs;
    sb->idx[warp] = bi;
    sb->pos[warp] = bp;
  }
  __syncthreads();
  bs = sb->key[0];
  bi = sb->idx[0];
  bp = sb->pos[0];
#pragma unroll
  for (int w = 1; w < 4; ++w)
    if (sb->pos[w] >= 0 && (bp < 0 || better(sb->key[w], sb->idx[w], bs, bi))) {
      bs = sb->key[w];
      bi = sb->idx[w];
      bp = sb->pos[w];
    }
  __syncthreads();
}

// stage 3: one block (128 threads) per query.
//   1. gather the (gallery row, approximate score) candidates of every segment slot of this query's q-tile
//   2. prune: with A_k the k-th largest approximate score, a candidate below A_k - 2*eps cannot be in the exact
//      top-k (its exact score is < A_k - eps <= the exact scores of the k best-approximate candidates)
//   3. exact fp64 scores of the survivors, selection by (score desc, index asc)
//   4. certificate against the rows the fused kernel dropped; failures are appended to `flagged` together with
//      a threshold for the second-chance pass (thr_next).
__global__ void __launch_bounds__(128)
    rescore_select_kernel(const float* __restrict__ q, const float* __restrict__ g, int nq, int ng, int d, int k,
                          int n_qtiles, int n_gtiles, int gchunk, int n_chunks, int n_units, int rows_per_qtile,
                          int n_sets, int d_pad, const uint2* __restrict__ cand, const int* __restrict__ cand_cnt,
                          const float* __restrict__ cand_thr, const int* __restrict__ qmap,
                          const float* __restrict__ mu, const float* __restrict__ nu, const int* __restrict__ nu_flag,
                          const float* __restrict__ q_norm_hat,
                          const float* __restrict__ q_norm_res, const float* __restrict__ q_norm_x,
                          const unsigned int* __restrict__ g_max,
                          long long g_index_base, long long g_index_stride, float* __restrict__ out_scores,
                          long long* __restrict__ out_idx, int* __restrict__ flagged, int* __restrict__ n_flagged,
                          float* __restrict__ thr_next, int max_cand) {
  extern __shared__ __align__(16) uint8_t sm[];
  double* qs = reinterpret_cast<double*>(sm);                          // [d] the query row, widened once
  double* sc = qs + ((d + 1) & ~1);                                    // [max_cand] scratch keys / exact scores
  int* ci = reinterpret_cast<int*>(sc + max_cand);                      // [max_cand] gallery rows of all candidates
  float* ap = reinterpret_cast<float*>(ci + max_cand);                  // [max_cand] approximate scores
  int* kc = reinterpret_cast<int*>(ap + max_cand);                      // [max_cand] gallery rows of the survivors
  __shared__ int s_n, s_overflow, s_kept, s_nslots, s_off[kMaxSlotsPerQuery], s_cnt[kMaxSlotsPerQuery], s_slot[kMaxSlotsPerQuery];
  __shared__ float s_thr, s_eps, s_qx, s_gn, s_ak, s_nun, s_mun;
  __shared__ double s_qmu, s_kth;
  __shared__ BlockBest s_bb;

  // blockIdx.x indexes the (possibly compacted) query matrix the fused kernel saw; qrow is the caller's row
  const int crow = blockIdx.x;
  const int qrow = qmap ? qmap[crow] : crow;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = threadIdx.x; c < d; c += blockDim.x) qs[c] = q[static_cast<size_t>(qrow) * d + c];

  const int qi = crow / rows_per_qtile, r = crow % rows_per_qtile;
  if (threadIdx.x == 0) {
    int n = 0, overflow = 0, ns = 0;
    float thr = -INFINITY;
    for (int c = 0; c < n_chunks; ++c) {      // mirror of SegWalker: which (chunk, unit) segments cover this q-tile
      const int g_lo = c * gchunk;
      const int ncg = min(gchunk, n_gtiles - g_lo);
      const long long T = static_cast<long long>(n_qtiles) * ncg;
      const long long u_lo = owner_unit(static_cast<long long>(qi) * ncg, T, n_units);
      const long long u_hi = owner_unit(static_cast<long long>(qi + 1) * ncg - 1, T, n_units);
      for (long long us = u_lo * n_sets; us < (u_hi + 1) * n_sets; ++us) {   // n_sets candidate slots per segment
        const int slot = (c * (n_units + n_qtiles) + static_cast<int>(us / n_sets) + qi) * n_sets + static_cast<int>(us % n_sets);
        const size_t sr = static_cast<size_t>(slot) * rows_per_qtile + r;
        int cc = cand_cnt[sr];
        thr = fmaxf(thr, cand_thr[sr]);
        if (n + cc > max_cand || ns >= kMaxSlotsPerQuery) {   // cannot happen with make_plan's bounds
          cc = 0;
          overflow = 1;
        }
        if (ns < kMaxSlotsPerQuery) {
          s_off[ns] = n;
          s_cnt[ns] = cc;
          s_slot[ns] = slot;
          ++ns;
        }
        n += cc;
      }
    }
    s_nslots = ns;
    s_n = n;
    s_thr = thr;
    s_overflow = overflow;
    s_kept = 0;
    // eps bounds |tensor-core score of (bf16 q, bf16 (g-mu)) - q.(g-mu)| for this query from the measured norms
    // (DESIGN.md section 4): bf16 rounding of both operands, fp32 accumulation, fp32 rounding of g - mu.
    const float g_norm = __uint_as_float(g_max[0]), g_res = __uint_as_float(g_max[1]);
    const float qh = q_norm_hat[qrow], qr = q_norm_res[qrow], qx = q_norm_x[qrow];
    s_eps = 1.001f * (qh * g_res + qr * g_norm) + d_pad * 2.4e-7f * qh * (g_norm + g_res) + 1e-30f;
    s_qx = qx;
    s_gn = g_norm;
  }
  __syncthreads();
  if (warp == 1) {   // ||nu||: fp32 roundings of q - nu, g - mu, the offset nu.(g - mu) and its addition
    float acc = 0.f;
    if (nu && nu_flag && *nu_flag)
      for (int c = lane; c < d; c += 32) acc += nu[c] * nu[c];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(kFull, acc, off);
    if (lane == 0) {
      s_nun = sqrtf(acc) * 1.001f;
      s_eps += 3e-7f * (s_qx + s_nun) * s_gn;
    }
  }
  if (warp == 0) {   // q . mu in fp64: the constant the centred approximate scores are offset by
    double acc = 0.0;
    float mu2 = 0.f;
    if (mu)
      for (int c = lane; c < d; c += 32) {
        acc = fma(qs[c], static_cast<double>(mu[c]), acc);
        mu2 = fmaf(mu[c], mu[c], mu2);
      }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      acc += __shfl_xor_sync(kFull, acc, off);
      mu2 += __shfl_xor_sync(kFull, mu2, off);
    }
    if (lane == 0) {
      s_qmu = acc;
      s_mun = sqrtf(mu2) * 1.001f;
    }
  }
  const int nslots = s_nslots;
  for (int t = threadIdx.x; t < nslots * kKPMax; t += blockDim.x) {
    const int s = t / kKPMax, j = t % kKPMax;
    if (j < s_cnt[s]) {
      const size_t sr = static_cast<size_t>(s_slot[s]) * rows_per_qtile + r;
      const uint2 e = cand[sr * kKPMax + j];
      ci[s_off[s] + j] = static_cast<int>(e.y);
      ap[s_off[s] + j] = __uint_as_float(e.x);
    }
  }
  __syncthreads();
  const int n = s_n;
  const int kk = min(k, n);

  // ---- prune by approximate score ----
  // A_k = k-th largest approximate score, found by rank counting (n is a few dozen: one pass, one barrier, instead of k
  // block-wide arg-max rounds)
  if (threadIdx.x == 0) s_ak = -INFINITY;
  __syncthreads();
  for (int c = threadIdx.x; c < n; c += blockDim.x) {
    const float v = ap[c];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const float o = ap[j];
      rank += (o > v) || (o == v && j < c);
    }
    if (rank == kk - 1) s_ak = v;
  }
  __syncthreads();
  const float a_k = s_ak;
  const float cut = a_k - 2.f * s_eps - 1e-6f * fabsf(a_k);
  for (int c = threadIdx.x; c < n; c += blockDim.x)
    if (n <= k || ap[c] >= cut) kc[atomicAdd(&s_kept, 1)] = ci[c];
  __syncthreads();
  const int m = s_kept;

  // ---- exact scores of the survivors, then selection by (score desc, index asc): again by rank counting ----
  for (int c = warp; c < m; c += 4) {
    const double v = exact_dot_warp_qd(qs, g + static_cast<size_t>(kc[c]) * d, d, lane);
    if (lane == 0) sc[c] = v;
  }
  if (threadIdx.x == 0) s_kth = -INFINITY;
  __syncthreads();
  const int km = min(k, m);
  for (int c = threadIdx.x; c < m; c += blockDim.x) {
    const double v = sc[c];
    const int iv = kc[c];
    int rank = 0;
    for (int j = 0; j < m; ++j) {
      const double o = sc[j];
      const int io = kc[j];
      rank += (o > v) || (o == v && (io < iv || (io == iv && j < c)));   // candidate rows are distinct; j < c only for safety
    }
    if (rank < km) {
      out_scores[static_cast<size_t>(qrow) * k + rank] = static_cast<float>(v);
      out_idx[static_cast<size_t>(qrow) * k + rank] = g_index_base + g_index_stride * iv;
      if (rank == km - 1) s_kth = v;
    }
  }
  __syncthreads();
  const double kth = (km > 0) ? s_kth : -INFINITY;
  if (threadIdx.x == 0) {
    // certificate: every gallery row g that is not a candidate has approximate centred score <= s_thr, hence exact
    // score q.g <= s_thr + eps + q.mu
    const bool closed = s_thr > -INFINITY;   // some segment dropped rows
    // fp64 rounding of kth and q.mu themselves (each a d-term dot of vectors no longer than (|q'| + |nu|), (|g'| + |mu|)):
    // irrelevant next to eps except when the centred gallery is (nearly) zero -- all rows identical -- and eps with it
    const double slack = 4.6e-16 * (d + 8) * static_cast<double>(s_qx + s_nun) * static_cast<double>(s_gn + s_mun);
    const bool ok = (n >= k) && (m >= k) && !s_overflow &&
                    (!closed || kth > static_cast<double>(s_thr) + static_cast<double>(s_eps) + s_qmu + slack);
    if (!ok) {
      const int pos = atomicAdd(n_flagged, 1);
      flagged[pos] = qrow;
      if (thr_next) {
        // every row of the true top-k has exact score >= kth, hence centred approximate score >= kth - q.mu - eps
        float t = -INFINITY;
        if (m >= k && kth > -INFINITY) {
          const double lo = kth - s_qmu - static_cast<double>(s_eps);
          t = static_cast<float>(lo) - 2e-6f * fabsf(static_cast<float>(lo)) - 1e-7f;
        }
        thr_next[pos] = t;
      }
    }
  }
}

// stage 3, one WARP per query (four queries per block, no block-wide barrier): the same steps and the same arithmetic
// as rescore_select_kernel -- identical candidate sets, eps, exact scores, order and certificate -- for passes whose
// q-tiles are covered by at most 32 candidate slots (a lane per slot; kKPMax = 32 entries per slot: a lane per entry).
// The block form spent a third of its warp time on barriers behind one thread's slot walk and fetched one gallery row
// per warp at a time: 171 us for 10k queries x ~14 surviving rows (1.7 TB/s of gathers).
constexpr int kRescoreWarps = 4;

// two rows, each with exactly the association of exact_dot_warp_qd; both rows' loads are issued before the first fma
DCR_DEVICE void exact_dot_warp_qd2(const double* __restrict__ a_smem, const float* __restrict__ b0,
                                   const float* __restrict__ b1, int d, uint32_t lane, double& out0, double& out1) {
  double acc0 = 0.0, acc1 = 0.0;
  if ((d & 127) == 0 && d <= 512) {
    // every lane owns d/128 whole 16-byte granules of each row: all (up to eight) loads are issued before the first fma --
    // written as a loop, each 128-column step waited for its own two loads (40 serial memory latencies per query)
    float4 v0[4], v1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i * 128 < d) {
        v0[i] = *reinterpret_cast<const float4*>(b0 + lane * 4 + i * 128);
        v1[i] = *reinterpret_cast<const float4*>(b1 + lane * 4 + i * 128);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i * 128 < d) {
        const double2 a01 = *reinterpret_cast<const double2*>(a_smem + lane * 4 + i * 128);
        const double2 a23 = *reinterpret_cast<const double2*>(a_smem + lane * 4 + i * 128 + 2);
        acc0 = fma(a01.x, static_cast<double>(v0[i].x), acc0);
        acc0 = fma(a01.y, static_cast<double>(v0[i].y), acc0);
        acc0 = fma(a23.x, static_cast<double>(v0[i].z), acc0);
        acc0 = fma(a23.y, static_cast<double>(v0[i].w), acc0);
        acc1 = fma(a01.x, static_cast<double>(v1[i].x), acc1);
        acc1 = fma(a01.y, static_cast<double>(v1[i].y), acc1);
        acc1 = fma(a23.x, static_cast<double>(v1[i].z), acc1);
        acc1 = fma(a23.y, static_cast<double>(v1[i].w), acc1);
      }
    }
  } else {
    for (int c = lane * 4; c < d; c += 128) {
      if (c + 3 < d) {
        const float4 v0 = *reinterpret_cast<const float4*>(b0 + c);
        const float4 v1 = *reinterpret_cast<const float4*>(b1 + c);
        const double2 a01 = *reinterpret_cast<const double2*>(a_smem + c);
        const double2 a23 = *reinterpret_cast<const double2*>(a_smem + c + 2);
        acc0 = fma(a01.x, static_cast<double>(v0.x), acc0);
        acc0 = fma(a01.y, static_cast<double>(v0.y), acc0);
        acc0 = fma(a23.x, static_cast<double>(v0.z), acc0);
        acc0 = fma(a23.y, static_cast<double>(v0.w), acc0);
        acc1 = fma(a01.x, static_cast<double>(v1.x), acc1);
        acc1 = fma(a01.y, static_cast<double>(v1.y), acc1);
        acc1 = fma(a23.x, static_cast<double>(v1.z), acc1);
        acc1 = fma(a23.y, static_cast<double>(v1.w), acc1);
      } else {
        for (int e = c; e < d; ++e) {
          acc0 = fma(a_smem[e], static_cast<double>(b0[e]), acc0);
          acc1 = fma(a_smem[e], static_cast<double>(b1[e]), acc1);
        }
      }
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    acc0 += __shfl_xor_sync(kFull, acc0, off);
    acc1 += __shfl_xor_sync(kFull, acc1, off);
  }
  out0 = acc0;
  out1 = acc1;
}

__global__ void __launch_bounds__(32 * kRescoreWarps)
    rescore_select_warp_kernel(const float* __restrict__ q, const float* __restrict__ g, int nq_pass, int d, int k,
                               int n_qtiles, int n_gtiles, int gchunk, int n_chunks, int n_units, int rows_per_qtile,
                               int n_sets, int d_pad, const uint2* __restrict__ cand, const int* __restrict__ cand_cnt,
                               const float* __restrict__ cand_thr, const int* __restrict__ qmap,
                               const float* __restrict__ mu, const float* __restrict__ nu, const int* __restrict__ nu_flag,
                               const float* __restrict__ q_norm_hat, const float* __restrict__ q_norm_res,
                               const float* __restrict__ q_norm_x, const unsigned int* __restrict__ g_max,
                               long long g_index_base, long long g_index_stride, float* __restrict__ out_scores,
                               long long* __restrict__ out_idx, int* __restrict__ flagged, int* __restrict__ n_flagged,
                               float* __restrict__ thr_next, int max_cand) {
  extern __shared__ __align__(16) uint8_t sm[];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int crow = blockIdx.x * kRescoreWarps + static_cast<int>(warp);
  if (crow >= nq_pass) return;   // whole warps leave; nothing below synchronises the block
  const int d2 = (d + 1) & ~1, mc = (max_cand + 3) & ~3;
  uint8_t* base = sm + static_cast<size_t>(warp) * (static_cast<size_t>(d2) * 8 + static_cast<size_t>(mc) * 20);
  double* qs = reinterpret_cast<double*>(base);     // [d2] the query row, widened once
  double* sc = qs + d2;                              // [mc] exact scores of the survivors
  int* ci = reinterpret_cast<int*>(sc + mc);         // [mc] gallery rows of all candidates
  float* ap = reinterpret_cast<float*>(ci + mc);     // [mc] approximate scores
  int* kc = reinterpret_cast<int*>(ap + mc);         // [mc] gallery rows of the survivors
  const int qrow = qmap ? qmap[crow] : crow;
  // the query row: requested first, consumed after the slot walk below has issued its own loads (one memory round trip for
  // both instead of one after the other)
  const bool q_fast = (d & 127) == 0 && d <= 512;
  float4 qv[4];
  if (q_fast) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (i * 128 < d) qv[i] = *reinterpret_cast<const float4*>(q + static_cast<size_t>(qrow) * d + lane * 4 + i * 128);
  }

  // ---- which (chunk, unit, set) slots cover this q-tile (mirror of SegWalker): lane c owns chunk c, then lane s slot s ----
  const int qi = crow / rows_per_qtile, r = crow % rows_per_qtile;
  int my_lo = 0, my_cnt = 0;
  if (static_cast<int>(lane) < n_chunks) {
    const int g_lo = lane * gchunk;
    const int ncg = min(gchunk, n_gtiles - g_lo);
    const long long T = static_cast<long long>(n_qtiles) * ncg;
    const long long u_lo = owner_unit(static_cast<long long>(qi) * ncg, T, n_units);
    const long long u_hi = owner_unit(static_cast<long long>(qi + 1) * ncg - 1, T, n_units);
    my_lo = static_cast<int>(u_lo);
    my_cnt = static_cast<int>(u_hi - u_lo + 1) * n_sets;
  }
  int ns = 0, my_slot = -1;
  for (int c = 0; c < n_chunks; ++c) {
    const int lo = __shfl_sync(kFull, my_lo, c), cnt = __shfl_sync(kFull, my_cnt, c);
    const int rel = static_cast<int>(lane) - ns;
    if (rel >= 0 && rel < cnt) my_slot = (c * (n_units + n_qtiles) + lo + rel / n_sets + qi) * n_sets + rel % n_sets;
    ns += cnt;
  }
  int cc = 0;
  float thr = -INFINITY;
  if (my_slot >= 0) {
    const size_t sr = static_cast<size_t>(my_slot) * rows_per_qtile + r;
    cc = cand_cnt[sr];
    thr = cand_thr[sr];
  }
  if (q_fast) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i * 128 < d) {
        double* dst = qs + lane * 4 + i * 128;
        *reinterpret_cast<double2*>(dst) = make_double2(static_cast<double>(qv[i].x), static_cast<double>(qv[i].y));
        *reinterpret_cast<double2*>(dst + 2) = make_double2(static_cast<double>(qv[i].z), static_cast<double>(qv[i].w));
      }
    }
  } else {
    for (int c = lane; c < d; c += 32) qs[c] = static_cast<double>(q[static_cast<size_t>(qrow) * d + c]);
  }
  int off = cc;   // inclusive prefix sum of the slot counts
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFull, off, o);
    if (static_cast<int>(lane) >= o) off += t;
  }
  const int n_total = __shfl_sync(kFull, off, 31);
  off -= cc;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) thr = fmaxf(thr, __shfl_xor_sync(kFull, thr, o));
  const bool overflow = ns > 32 || n_total > max_cand;   // cannot happen: the host picks this kernel for <= 32 slots
  const int n = overflow ? 0 : n_total;
  const int nsl = min(ns, 32);
#pragma unroll 4
  for (int s = 0; s < nsl; ++s) {
    const int c_s = overflow ? 0 : __shfl_sync(kFull, cc, s), off_s = __shfl_sync(kFull, off, s);
    const int slot_s = __shfl_sync(kFull, my_slot, s);
    if (static_cast<int>(lane) < c_s) {
      const uint2 e = cand[(static_cast<size_t>(slot_s) * rows_per_qtile + r) * kKPMax + lane];
      ci[off_s + lane] = static_cast<int>(e.y);
      ap[off_s + lane] = __uint_as_float(e.x);
    }
  }

  // eps bounds |tensor-core score of (bf16 q, bf16 (g-mu)) - q.(g-mu)| for this query from the measured norms
  // (DESIGN.md section 4); same expression, same order of operations as the block form
  const float g_norm = __uint_as_float(g_max[0]), g_res = __uint_as_float(g_max[1]);
  const float qh = q_norm_hat[qrow], qr = q_norm_res[qrow], qx = q_norm_x[qrow];
  float eps = 1.001f * (qh * g_res + qr * g_norm) + d_pad * 2.4e-7f * qh * (g_norm + g_res) + 1e-30f;
  float nun = 0.f, mun = 0.f;   // |nu|, |mu| (upper bounds)
  {
    float acc = 0.f;
    if (nu && nu_flag && *nu_flag)
      for (int c = lane; c < d; c += 32) acc += nu[c] * nu[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
    nun = sqrtf(acc) * 1.001f;
    eps += 3e-7f * (qx + nun) * g_norm;
  }
  __syncwarp();
  double qmu = 0.0;   // q . mu in fp64: the constant the centred approximate scores are offset by
  if (mu) {
    float mu2 = 0.f;
    for (int c = lane; c < d; c += 32) {
      qmu = fma(qs[c], static_cast<double>(mu[c]), qmu);
      mu2 = fmaf(mu[c], mu[c], mu2);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      qmu += __shfl_xor_sync(kFull, qmu, o);
      mu2 += __shfl_xor_sync(kFull, mu2, o);
    }
    mun = sqrtf(mu2) * 1.001f;
  }

  // ---- prune by approximate score: A_k by rank counting ----
  const int kk = min(k, n);
  float a_k = -INFINITY;
  for (int c = lane; c < n; c += 32) {
    const float v = ap[c];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const float o = ap[j];
      rank += (o > v) || (o == v && j < c);
    }
    if (rank == kk - 1) a_k = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a_k = fmaxf(a_k, __shfl_xor_sync(kFull, a_k, o));
  const float cut = a_k - 2.f * eps - 1e-6f * fabsf(a_k);
  int m = 0;
  for (int c0 = 0; c0 < n; c0 += 32) {
    const int c = c0 + lane;
    const bool keep = c < n && (n <= k || ap[c] >= cut);
    const uint32_t mask = __ballot_sync(kFull, keep);
    if (keep) kc[m + __popc(mask & ((1u << lane) - 1u))] = ci[c];
    m += __popc(mask);
  }
  __syncwarp();
  // every surviving row's cache lines are requested at once (L2 prefetch): the dot products below then wait for L2, not for
  // one DRAM round trip per pair of rows
  {
    const int lines = (d * 4 + 127) / 128;
    for (int t = lane; t < m * lines; t += 32) {
      const float* ptr = g + static_cast<size_t>(kc[t / lines]) * d + (t % lines) * 32;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr));
    }
  }

  // ---- exact scores of the survivors (two rows in flight), then selection by (score desc, index asc) ----
  for (int c = 0; c < m; c += 2) {
    double v0, v1 = 0.0;
    if (c + 1 < m) exact_dot_warp_qd2(qs, g + static_cast<size_t>(kc[c]) * d, g + static_cast<size_t>(kc[c + 1]) * d, d, lane, v0, v1);
    else v0 = exact_dot_warp_qd(qs, g + static_cast<size_t>(kc[c]) * d, d, lane);
    if (lane == 0) {
      sc[c] = v0;
      if (c + 1 < m) sc[c + 1] = v1;
    }
  }
  __syncwarp();
  const int km = min(k, m);
  double kth = -INFINITY;
  for (int c = lane; c < m; c += 32) {
    const double v = sc[c];
    const int iv = kc[c];
    int rank = 0;
    for (int j = 0; j < m; ++j) {
      const double o = sc[j];
      const int io = kc[j];
      rank += (o > v) || (o == v && (io < iv || (io == iv && j < c)));
    }
    if (rank < km) {
      out_scores[static_cast<size_t>(qrow) * k + rank] = static_cast<float>(v);
      out_idx[static_cast<size_t>(qrow) * k + rank] = g_index_base + g_index_stride * iv;
      if (rank == km - 1) kth = v;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kth = fmax(kth, __shfl_xor_sync(kFull, kth, o));   // one lane holds it (NaN -> -inf: flagged)
  if (lane == 0) {
    // certificate: every gallery row that is not a candidate has approximate centred score <= thr, hence exact score
    // q.g <= thr + eps + q.mu
    const bool closed = thr > -INFINITY;
    // fp64 rounding of kth and q.mu themselves: see the block form
    const double slack = 4.6e-16 * (d + 8) * static_cast<double>(qx + nun) * static_cast<double>(g_norm + mun);
    const bool ok = (n >= k) && (m >= k) && !overflow &&
                    (!closed || kth > static_cast<double>(thr) + static_cast<double>(eps) + qmu + slack);
    if (!ok) {
      const int pos = atomicAdd(n_flagged, 1);
      flagged[pos] = qrow;
      if (thr_next) {
        float t = -INFINITY;
        if (m >= k && kth > -INFINITY) {
          const double lo = kth - qmu - static_cast<double>(eps);
          t = static_cast<float>(lo) - 2e-6f * fabsf(static_cast<float>(lo)) - 1e-7f;
        }
        thr_next[pos] = t;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// 'splitloss' similarity (diff_retrieval.py:393-400): descriptors are cut into n_chunks equal parts and the score of
// a pair is the MAXIMUM over the parts of the per-part dot products.  The top-k under that score is contained in the
// union of the per-part top-k lists (if a row is in the true top-k through its best part c, fewer than k rows beat it
// in part c), so the host runs the fused kernel once per part and this kernel finishes: per query, de-duplicate the
// n_cand candidate rows, evaluate max_c <q_c, g_c> exactly (float64, the same fixed-order dot as the re-score
// kernel), and select k by (score desc, row asc).
__global__ void __launch_bounds__(128)
    split_rescore_kernel(const float* __restrict__ q, const float* __restrict__ g, int d, int n_chunks, int cross,
                         const long long* __restrict__ cand, int n_cand, int k, float* __restrict__ out_scores,
                         long long* __restrict__ out_idx) {
  extern __shared__ __align__(16) uint8_t sm[];
  // only ONE query part is staged at a time (per-token splitloss on ViT outputs has d = 197 * 384 floats per row)
  const int p = d / n_chunks;
  float* qs = reinterpret_cast<float*>(sm);                              // [p]
  double* sc = reinterpret_cast<double*>(sm + ((p * 4 + 15) & ~15));      // [n_cand]
  long long* ci = reinterpret_cast<long long*>(sc + n_cand);              // [n_cand], -1 = duplicate / taken
  __shared__ BlockBest s_bb;
  const int qrow = blockIdx.x;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = threadIdx.x; c < n_cand; c += blockDim.x) ci[c] = cand[static_cast<size_t>(qrow) * n_cand + c];
  __syncthreads();
  // duplicates (a row that made the list of several parts): keep the first occurrence
  for (int c = threadIdx.x; c < n_cand; c += blockDim.x) {
    const long long v = ci[c];
    bool dup = v < 0;                                                     // negative = empty slot of the caller's list
    for (int j = 0; j < c; ++j) dup |= (ci[j] == v);   // ci is not modified before the barrier below
    sc[c] = dup ? 1.0 : 0.0;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < n_cand; c += blockDim.x) {
    if (sc[c] != 0.0) ci[c] = -1;
    sc[c] = -INFINITY;
  }
  __syncthreads();
  for (int qp = 0; qp < n_chunks; ++qp) {
    for (int c = threadIdx.x; c < p; c += blockDim.x) qs[c] = q[static_cast<size_t>(qrow) * d + qp * p + c];
    __syncthreads();
    for (int c = warp; c < n_cand; c += 4) {
      if (ci[c] < 0) continue;   // warp-uniform
      double best = sc[c];
      if (cross) {   // 'cross' (einsum_in_chunks, diff_retrieval.py:652-654): every gallery part against every query part
        for (int part = 0; part < n_chunks; ++part)
          best = fmax(best, exact_dot_warp(qs, g + static_cast<size_t>(ci[c]) * d + part * p, p, lane));
      } else {
        best = fmax(best, exact_dot_warp(qs, g + static_cast<size_t>(ci[c]) * d + qp * p, p, lane));
      }
      if (lane == 0) sc[c] = best;   // ranked on the float64 value (as dcr_sim_topk), reported as fp32
    }
    __syncthreads();
  }
  for (int round = 0; round < k; ++round) {
    double bs = -INFINITY;
    long long bi = 0x7fffffffffffffffLL;
    int bp = -1;
    for (int c = threadIdx.x; c < n_cand; c += blockDim.x)
      if (ci[c] >= 0 && (bp < 0 || better(sc[c], ci[c], bs, bi))) {
        bs = sc[c];
        bi = ci[c];
        bp = c;
      }
    block_argbest(bs, bi, bp, &s_bb, lane, warp);
    if (threadIdx.x == 0) {
      out_scores[static_cast<size_t>(qrow) * k + round] = bp >= 0 ? static_cast<float>(bs) : -INFINITY;
      out_idx[static_cast<size_t>(qrow) * k + round] = bp >= 0 ? bi : -1;
      if (bp >= 0) ci[bp] = -1;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------------------
// brute-force exact path for flagged queries (batch of <= kExactBatch): scores[f][g] in fp64, then select.
constexpr int kExactBatch = 32;

__global__ void __launch_bounds__(256)
    exact_scan_kernel(const float* __restrict__ q, const float* __restrict__ g, int ng, int d,
                      const int* __restrict__ flagged, int f_begin, const int* __restrict__ n_flagged,
                      double* __restrict__ scores, int batch) {
  extern __shared__ __align__(16) uint8_t sm[];
  float* qs = reinterpret_cast<float*>(sm);  // [nb][d]
  const int nb = min(batch, *n_flagged - f_begin);
  if (nb <= 0) return;
  for (int i = threadIdx.x; i < nb * d; i += blockDim.x) {
    const int f = i / d, c = i % d;
    qs[i] = q[static_cast<size_t>(flagged[f_begin + f]) * d + c];
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const int warps = (blockDim.x >> 5) * gridDim.x;
  for (int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < ng; row += warps) {
    const float* gr = g + static_cast<size_t>(row) * d;
    for (int f = 0; f < nb; ++f) {
      const double v = exact_dot_warp(qs + f * d, gr, d, lane);
      if (lane == 0) scores[static_cast<size_t>(f) * ng + row] = v;
    }
  }
}

__global__ void __launch_bounds__(256)
    exact_select_kernel(double* __restrict__ scores, int ng, int k, const int* __restrict__ flagged, int f_begin,
                        const int* __restrict__ n_flagged, long long g_index_base, long long g_index_stride,
                        float* __restrict__ out_scores, long long* __restrict__ out_idx) {
  const int f = blockIdx.x;
  if (f_begin + f >= *n_flagged) return;
  const int qrow = flagged[f_begin + f];
  double* s = scores + static_cast<size_t>(f) * ng;
  __shared__ double s_best[8];
  __shared__ int s_besti[8];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int round = 0; round < k; ++round) {
    double bs = -INFINITY;
    int bi = -1;
    for (int c = threadIdx.x; c < ng; c += blockDim.x) {
      const double v = s[c];
      if (!(v != v) && (bi < 0 || v > bs)) {   // ascending c per thread => first (lowest index) max kept
        bs = v;
        bi = c;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const double os = __shfl_xor_sync(kFull, bs, off);
      const int oi = __shfl_xor_sync(kFull, bi, off);
      if (oi >= 0 && (bi < 0 || os > bs || (os == bs && oi < bi))) {
        bs = os;
        bi = oi;
      }
    }
    if (lane == 0) {
      s_best[warp] = bs;
      s_besti[warp] = bi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < 8; ++w)
        if (s_besti[w] >= 0 && (s_besti[0] < 0 || s_best[w] > s_best[0] ||
                                (s_best[w] == s_best[0] && s_besti[w] < s_besti[0]))) {
          s_best[0] = s_best[w];
          s_besti[0] = s_besti[w];
        }
      if (s_besti[0] < 0) {   // every remaining score is NaN (NaN query row, or k > number of non-NaN scores)
        out_scores[static_cast<size_t>(qrow) * k + round] = __int_as_float(0x7fc00000);
        out_idx[static_cast<size_t>(qrow) * k + round] = -1;
      } else {
        out_scores[static_cast<size_t>(qrow) * k + round] = static_cast<float>(s_best[0]);
        out_idx[static_cast<size_t>(qrow) * k + round] = g_index_base + g_index_stride * s_besti[0];
        s[s_besti[0]] = __longlong_as_double(0x7ff8000000000000LL);  // NaN marks "taken"
      }
    }
    __syncthreads();
  }
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// launch geometry of one fused pass over nq queries
struct PassPlan {
  int nq, nq_pad, n_qtiles, n_units, n_slots, kp, cap, stages, max_cand;
  int n_sets;             // epilogue warp sets = candidate slots per segment (column halves with their own lists)
  int gchunk, n_chunks;   // gallery tiles per L2-sized chunk for this pass
  size_t smem_bytes;
};

struct SimPlan {
  int d_pad, num_kb, ng_pad, n_gtiles, rows_per_qtile;
  int stream_a;  // d_pad > 512: query tile streamed with the gallery k-blocks
  int max_sets;  // upper bound for PassPlan::n_sets (1 or 2)
  int gchunk, n_chunks;   // preferred gallery chunking (a pass may use fewer chunks)
  int kp0, kp1;           // candidates kept by the first pass / by the second-chance pass (0 = no second pass)
  PassPlan p0, p1;        // p1 is sized for the worst case (every query flagged)
  // workspace offsets
  size_t off_qb, off_qb1, off_gb, off_qnh, off_qnr, off_qnx, off_gmax, off_colsum, off_mu, off_cand, off_cnt, off_thr,
      off_flag0, off_flag1, off_thr1, off_counts, off_exact, off_nu, off_bias, off_clk, off_gthr;
  size_t total;
};

int plan_pass(int nq, int kp, const SimPlan& sp, int num_sms, size_t max_smem, int d, int k, PassPlan* pp) {
  pp->nq = nq;
  pp->n_qtiles = (nq + sp.rows_per_qtile - 1) / sp.rows_per_qtile;
  pp->nq_pad = pp->n_qtiles * sp.rows_per_qtile;
  pp->kp = kp;
  // ---- shared memory: resident A + stages*B + n_sets * cap KB of lists + barriers + carried thresholds ----
  const size_t a_bytes = sp.stream_a ? 0 : static_cast<size_t>(sp.num_kb) * kATileBytes;
  const size_t b_tile = static_cast<size_t>(kBlockN / kCG) * kBlockK * 2 + (sp.stream_a ? kATileBytes : 0);
  const size_t fixed = 1024 /*align slack*/ + 256 /*barriers*/ + 4096 /*carried thresholds*/;
  auto fits = [&](int st, int cp, int sets) {
    return max_smem >= a_bytes + st * b_tile + static_cast<size_t>(cp) * 1024 * sets + fixed;
  };
  // two epilogue warp sets whenever their lists (at least kp + 8 entries per row and set) fit next to 3 B stages
  int sets = (sp.max_sets >= 2 && fits(3, kp + 8, 2)) ? 2 : 1;
  int cap = kp + (sets == 2 ? 8 : 16);
  int stages = 2;
  DCR_REQUIRE(fits(stages, cap, sets), "sim_topk: not enough shared memory (%zu B) for d=%d k=%d", max_smem, d, k);
  // priorities: 3 B stages, then list capacity up to 64 (fewer compactions), then more stages (up to 8)
  if (fits(3, cap, sets)) stages = 3;
  while (cap < 64 && fits(stages, cap + 1, sets)) ++cap;
  while (stages < 8 && fits(stages + 1, cap, sets)) ++stages;
  pp->cap = cap;
  pp->stages = stages;
  pp->n_sets = sets;
  pp->smem_bytes = fixed + a_bytes + stages * b_tile + static_cast<size_t>(cap) * 1024 * sets;

  // ---- gallery chunking and work units ----
  pp->gchunk = sp.gchunk;
  pp->n_chunks = sp.n_chunks;
  int units = 1;
  long long span_total = 0;
  for (;;) {
    const long long T = static_cast<long long>(pp->n_qtiles) * pp->gchunk;   // tiles of one (full) gallery chunk
    units = num_sms / kCG;
    if (T < units) units = static_cast<int>(std::max<long long>(1, T));
    // per chunk a q-tile is covered by at most ceil(tiles_in_chunk / (T_c / units)) + 1 units
    span_total = 0;
    for (int c = 0; c < pp->n_chunks; ++c) {
      const int ncg = std::min(pp->gchunk, sp.n_gtiles - c * pp->gchunk);
      const long long Tc = static_cast<long long>(pp->n_qtiles) * ncg;
      const long long per_unit = std::max<long long>(1, Tc / units);
      long long span = (ncg + per_unit - 1) / per_unit + 1;
      if (span > units) span = units;
      span_total += span * sets;
    }
    // the re-score kernel keeps every candidate of a query in shared memory (20 B each): few queries spread over all
    // units and many chunks would not fit -> use fewer chunks for such a pass
    if (pp->n_chunks == 1 || (span_total <= kMaxSlotsPerQuery && span_total * kp * 20 <= 150 * 1024)) break;
    pp->n_chunks = (pp->n_chunks + 1) / 2;
    pp->gchunk = (sp.n_gtiles + pp->n_chunks - 1) / pp->n_chunks;
    pp->n_chunks = (sp.n_gtiles + pp->gchunk - 1) / pp->gchunk;
  }
  pp->n_units = units;
  pp->n_slots = pp->n_chunks * (units + pp->n_qtiles) * sets;
  DCR_REQUIRE(span_total <= kMaxSlotsPerQuery, "sim_topk: %lld candidate slots per query tile (max %d)", span_total,
              kMaxSlotsPerQuery);
  pp->max_cand = static_cast<int>(span_total) * kp;
  return 0;
}

int make_plan(int nq, int ng, int d, int k, int num_sms, size_t max_smem, SimPlan* pl) {
  DCR_REQUIRE(nq >= 1 && ng >= 1 && d >= 1, "sim_topk: empty problem (nq=%d ng=%d d=%d)", nq, ng, d);
  DCR_REQUIRE(d <= kMaxDim, "sim_topk: descriptor dim %d > %d not supported", d, kMaxDim);
  DCR_REQUIRE(k >= 1 && k <= 16, "sim_topk: k=%d outside [1,16]", k);
  DCR_REQUIRE(k <= ng, "sim_topk: k=%d > gallery size %d", k, ng);
  pl->d_pad = static_cast<int>(align_up(d, kBlockK));
  pl->num_kb = pl->d_pad / kBlockK;
  pl->stream_a = pl->num_kb > kMaxKB ? 1 : 0;
  pl->rows_per_qtile = kBlockM * kCG;
  // Two epilogue warp sets (two warps per TMEM lane quadrant, each with its own lists for one column half) pay off when
  // few candidates are kept: measured on B200 (10k x 100k x 512) k = 1: 0.79 ms vs 0.82 ms and no second-chance pass
  // (each segment keeps 2 x 4 candidates); k = 10: slower (the lists of two sets only fit with a small capacity).
  pl->max_sets = k <= 2 ? 2 : 1;
  pl->n_gtiles = (ng + kBlockN - 1) / kBlockN;
  pl->ng_pad = pl->n_gtiles * kBlockN;
  // gallery chunks of ~40 MB of bf16 rows: the units sweep one chunk at a time so that it stays L2 resident
  const long long chunk_bytes = 40ll << 20;
  int gchunk = static_cast<int>(std::max<long long>(16, chunk_bytes / (static_cast<long long>(kBlockN) * pl->d_pad * 2)));
  int n_chunks = (pl->n_gtiles + gchunk - 1) / gchunk;
  if (n_chunks > 64) n_chunks = 64;
  gchunk = (pl->n_gtiles + n_chunks - 1) / n_chunks;   // equal chunks
  n_chunks = (pl->n_gtiles + gchunk - 1) / gchunk;
  pl->gchunk = gchunk;
  pl->n_chunks = n_chunks;
  // first pass keeps few candidates per (query, segment) -- enough unless many gallery rows sit within the error
  // bound of the k-th score; such queries get a second chance with 32 candidates before the brute-force path
  // k in 6..10 keeps 12 (measured on B200, 10k x 100k x 512, k = 10: 1.20 ms with 16, 1.14 ms with 12, 1.10 ms with 10;
  // two spare candidates per segment keep the second-chance pass rare)
  const int kp0 = (k <= 2) ? 4 : (k <= 5 ? 8 : (k <= 10 ? 12 : 32));
  DCR_REQUIRE(kp0 >= k, "sim_topk: first-pass candidate count %d < k=%d", kp0, k);
  pl->kp0 = kp0;
  pl->kp1 = (kp0 < kKPMax) ? kKPMax : 0;
  if (int rc = plan_pass(nq, pl->kp0, *pl, num_sms, max_smem, d, k, &pl->p0)) return rc;
  if (pl->kp1) {
    if (plan_pass(nq, pl->kp1, *pl, num_sms, max_smem, d, k, &pl->p1) != 0) pl->kp1 = 0;   // does not fit: skip
  }
  const PassPlan& big = pl->p0;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  pl->off_qb = take(static_cast<size_t>(big.nq_pad) * pl->d_pad * 2);
  pl->off_qb1 = take(pl->kp1 ? static_cast<size_t>(pl->p1.nq_pad) * pl->d_pad * 2 : 0);
  pl->off_gb = take(static_cast<size_t>(pl->ng_pad) * pl->d_pad * 2);
  pl->off_qnh = take(static_cast<size_t>(big.nq_pad) * 4);
  pl->off_qnr = take(static_cast<size_t>(big.nq_pad) * 4);
  pl->off_qnx = take(static_cast<size_t>(big.nq_pad) * 4);
  pl->off_gmax = take(16);
  pl->off_colsum = take(static_cast<size_t>(d) * 16);   // column sums + column sums of squares
  pl->off_mu = take(static_cast<size_t>(d) * 4);
  pl->off_nu = take(static_cast<size_t>(d) * 4);
  pl->off_bias = take(static_cast<size_t>(pl->ng_pad) * 4);
  const size_t slot_rows = static_cast<size_t>(std::max(pl->p0.n_slots, pl->kp1 ? pl->p1.n_slots : 0)) * pl->rows_per_qtile;   // n_slots counts sets
  pl->off_cand = take(slot_rows * kKPMax * 8);
  pl->off_cnt = take(slot_rows * 4);
  pl->off_thr = take(slot_rows * 4);
  pl->off_flag0 = take(static_cast<size_t>(nq) * 4);
  pl->off_flag1 = take(static_cast<size_t>(nq) * 4);
  pl->off_thr1 = take(static_cast<size_t>(nq) * 4);
  pl->off_counts = take(16);
  pl->off_clk = take(32);
  pl->off_gthr = take(static_cast<size_t>(std::max(big.nq_pad, pl->kp1 ? pl->p1.nq_pad : 0)) * 4);
  pl->off_exact = take(static_cast<size_t>(kExactBatch) * ng * 8);
  pl->total = off;
  return 0;
}

struct PassBuffers {
  uint2* cand;
  int* ccnt;
  float* cthr;
};

// one fused pass: qb (bf16, padded) x gb (bf16, centred, padded) -> candidate slots
int launch_fused(const SimPlan& pl, const PassPlan& pp, const __nv_bfloat16* qb, const __nv_bfloat16* gb, int ng,
                 const PassBuffers& pb, const float* col_bias, const int* bias_flag, const float* thr_init,
                 unsigned long long* clk, unsigned int* gthr, cudaStream_t stream) {
  CUtensorMap tq, tg;
  if (int rc = make_tmap_2d_bf16(&tq, qb, pp.nq_pad, pl.d_pad, pl.d_pad, kBlockM, kBlockK)) return rc;
  if (int rc = make_tmap_2d_bf16(&tg, gb, pl.ng_pad, pl.d_pad, pl.d_pad, kBlockN / kCG, kBlockK)) return rc;
  SimParams p;
  p.nq = pp.nq;
  p.ng = ng;
  p.num_kb = pl.num_kb;
  p.stream_a = pl.stream_a;
  p.n_qtiles = pp.n_qtiles;
  p.n_gtiles = pl.n_gtiles;
  p.gchunk = pp.gchunk;
  p.n_chunks = pp.n_chunks;
  p.kp = pp.kp;
  p.cap = pp.cap;
  p.stages = pp.stages;
  p.cand = pb.cand;
  p.cand_cnt = pb.ccnt;
  p.cand_thr = pb.cthr;
  p.col_bias = col_bias;
  p.bias_flag = bias_flag;
  p.thr_init = thr_init;
  p.clk = clk;
  p.gthr = gthr;
  DCR_CUDA_CHECK(cudaMemsetAsync(gthr, 0, static_cast<size_t>(pp.nq_pad) * 4, stream));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pp.n_units * kCG);
  cfg.blockDim = dim3(64 + 128 * pp.n_sets);
  cfg.dynamicSmemBytes = pp.smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  auto launch = [&](auto kern) -> int {
    DCR_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pp.smem_bytes)));
    DCR_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, tq, tg, p));
    count_launch();
    return 0;
  };
  // both variants are launched; the one that does not match the device flag of query centring returns at once
  if (pp.n_sets == 2) {
    if (int rc = launch(sim_topk_kernel<false, 2>)) return rc;
    return launch(sim_topk_kernel<true, 2>);
  }
  if (int rc = launch(sim_topk_kernel<false, 1>)) return rc;
  return launch(sim_topk_kernel<true, 1>);
}

}  // namespace

int split_rescore(const float* q, const float* g, int nq, int d, int n_chunks, int cross, const long long* cand, int n_cand,
                  int k, float* out_scores, long long* out_idx, cudaStream_t stream) {
  DCR_REQUIRE(nq >= 1 && d >= 1 && n_chunks >= 1 && d % n_chunks == 0 && (d / n_chunks) % 4 == 0,
              "split_rescore: d=%d must split into %d parts whose length is a multiple of 4", d, n_chunks);
  DCR_REQUIRE(n_cand >= k && k >= 1 && n_cand <= 4096, "split_rescore: need k <= n_cand <= 4096 (k=%d n_cand=%d)", k, n_cand);
  DCR_REQUIRE((reinterpret_cast<uintptr_t>(q) & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0,
              "split_rescore: q/g must be 16-byte aligned");
  const size_t smem = ((static_cast<size_t>(d / n_chunks) * 4 + 15) & ~size_t(15)) + static_cast<size_t>(n_cand) * 16;
  DCR_CUDA_CHECK(cudaFuncSetAttribute(split_rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  split_rescore_kernel<<<nq, 128, smem, stream>>>(q, g, d, n_chunks, cross, cand, n_cand, k, out_scores, out_idx);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

size_t sim_topk_workspace_size(int nq, int ng, int d, int k) {
  const DeviceInfo* di = device_info();
  SimPlan pl;
  if (make_plan(nq, ng, d, k, di ? di->num_sms : 148, di ? di->max_smem_optin : 232448, &pl) != 0)
    return 0;
  return pl.total;
}

int sim_topk(const float* q, int nq, const float* g, int ng, int d, int k, long long g_index_base,
             long long g_index_stride, float* out_scores, long long* out_idx, void* ws, size_t ws_bytes,
             cudaStream_t stream, SimStats* stats) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(di->cc_major == 10, "sim_topk: this build targets sm_100a; device reports sm_%d%d", di->cc_major, di->cc_minor);
  SimPlan pl;
  if (int rc = make_plan(nq, ng, d, k, di->num_sms, di->max_smem_optin, &pl)) return rc;
  DCR_REQUIRE(ws != nullptr && ws_bytes >= pl.total, "sim_topk: workspace too small (%zu < %zu)", ws_bytes, pl.total);
  DCR_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "sim_topk: workspace must be 256-byte aligned");
  DCR_REQUIRE((reinterpret_cast<uintptr_t>(q) & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0 && d % 4 == 0,
              "sim_topk: q/g must be 16-byte aligned with d %% 4 == 0 (d=%d)", d);
  uint8_t* w = static_cast<uint8_t*>(ws);
  auto* qb = reinterpret_cast<__nv_bfloat16*>(w + pl.off_qb);
  auto* qb1 = reinterpret_cast<__nv_bfloat16*>(w + pl.off_qb1);
  auto* gb = reinterpret_cast<__nv_bfloat16*>(w + pl.off_gb);
  auto* qnh = reinterpret_cast<float*>(w + pl.off_qnh);
  auto* qnr = reinterpret_cast<float*>(w + pl.off_qnr);
  auto* qnx = reinterpret_cast<float*>(w + pl.off_qnx);
  auto* gmax = reinterpret_cast<unsigned int*>(w + pl.off_gmax);
  auto* colsum = reinterpret_cast<double*>(w + pl.off_colsum);
  auto* mu = reinterpret_cast<float*>(w + pl.off_mu);
  auto* nu = reinterpret_cast<float*>(w + pl.off_nu);
  auto* bias = reinterpret_cast<float*>(w + pl.off_bias);
  PassBuffers pb;
  pb.cand = reinterpret_cast<uint2*>(w + pl.off_cand);
  pb.ccnt = reinterpret_cast<int*>(w + pl.off_cnt);
  pb.cthr = reinterpret_cast<float*>(w + pl.off_thr);
  auto* flag0 = reinterpret_cast<int*>(w + pl.off_flag0);
  auto* flag1 = reinterpret_cast<int*>(w + pl.off_flag1);
  auto* thr1 = reinterpret_cast<float*>(w + pl.off_thr1);
  auto* counts = reinterpret_cast<int*>(w + pl.off_counts);   // [0] flagged by pass 0, [1] flagged by pass 1
  auto* exact = reinterpret_cast<double*>(w + pl.off_exact);
  auto* clk = reinterpret_cast<unsigned long long*>(w + pl.off_clk);
  auto* gthr = reinterpret_cast<unsigned int*>(w + pl.off_gthr);

  DCR_CUDA_CHECK(cudaMemsetAsync(gmax, 0, 16, stream));
  DCR_CUDA_CHECK(cudaMemsetAsync(counts, 0, 16, stream));   // [0],[1] flagged counts, [2] query-centring flag
  const int conv_blocks = di->num_sms * 8;
  int* qflag = counts + 2;   // device flag: query centring on/off
  auto sampled_mean = [&](const float* x, int n, float* out, bool decide) -> int {
    // any fixed vector works as a centre, so a strided sample of <= 8192 rows is enough
    DCR_CUDA_CHECK(cudaMemsetAsync(colsum, 0, static_cast<size_t>(d) * 16, stream));
    const int row_stride = std::max(1, n / 8192);
    const int n_sample = (n + row_stride - 1) / row_stride;
    col_sum_kernel<<<std::max(1, std::min((n_sample + 63) / 64, di->num_sms)), kColSumThreads, 0, stream>>>(
        x, n_sample, row_stride, d, colsum, decide ? colsum + d : nullptr);
    count_launch();
    col_mean_finish_kernel<<<(d + 255) / 256, 256, 0, stream>>>(colsum, n_sample, d, out);
    count_launch();
    if (decide) {
      centre_decision_kernel<<<1, 256, 0, stream>>>(colsum, colsum + d, n_sample, d, qflag);
      count_launch();
    }
    return 0;
  };
  if (int rc = sampled_mean(g, ng, mu, false)) return rc;    // gallery centre mu (always used)
  if (int rc = sampled_mean(q, nq, nu, true)) return rc;     // query centre nu + the decision whether to use it
  // q' = q - nu, g' = g - mu:  q.g = q'.g' + nu.g' + q.mu  -- the tensor cores see only the centred parts, nu.g' is a
  // per-gallery-row offset added to the accumulator columns, q.mu a per-query constant that cannot change the ranking
  // d_pad <= 256: 2 loads per lane cover the row; otherwise 4 per round (512 dims = one round)
  auto convert = (pl.d_pad <= 256) ? to_bf16_rows_kernel<2> : to_bf16_rows_kernel<4>;
  convert<<<conv_blocks, 256, 0, stream>>>(q, nq, d, pl.p0.nq_pad, pl.d_pad, nu, qb, qnh, qnr, qnx, nullptr,
                                           nullptr, nullptr, qflag, nullptr);
  count_launch();
  convert<<<conv_blocks, 256, 0, stream>>>(g, ng, d, pl.ng_pad, pl.d_pad, mu, gb, nullptr, nullptr, nullptr,
                                           gmax, nu, bias, nullptr, qflag);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());

  // CUDA events around the first fused pass only (thread-local, created once): bench.py's roofline numerator
  // (events belong to the device that was current when they were created: one pair per device)
  static thread_local cudaEvent_t ev_tab[64][2] = {};
  cudaEvent_t& ev0 = ev_tab[di->device][0];
  cudaEvent_t& ev1 = ev_tab[di->device][1];
  if (!ev0) {
    DCR_CUDA_CHECK(cudaEventCreate(&ev0));
    DCR_CUDA_CHECK(cudaEventCreate(&ev1));
  }
  DCR_CUDA_CHECK(cudaEventRecord(ev0, stream));
  if (int rc = launch_fused(pl, pl.p0, qb, gb, ng, pb, bias, qflag, nullptr, clk, gthr, stream)) return rc;
  DCR_CUDA_CHECK(cudaEventRecord(ev1, stream));

  auto rescore = [&](const PassPlan& pp, const int* qmap, int* flagged, int* n_flagged, float* thr_next) -> int {
    // one warp per query when a q-tile's candidate slots fit a lane each and four queries' rows fit a block's shared memory
    const size_t per_warp = ((static_cast<size_t>(d) + 1) & ~size_t(1)) * 8 + ((static_cast<size_t>(pp.max_cand) + 3) & ~size_t(3)) * 20;
    const bool warp_form = pp.kp > 0 && pp.max_cand / pp.kp <= 32 && pp.n_chunks <= 32 && kRescoreWarps * per_warp <= 56 * 1024 &&
                           !tuning_flag("DCR_SIM_RESCORE_BLOCK");
    if (warp_form) {
      const size_t smem = kRescoreWarps * per_warp;
      DCR_CUDA_CHECK(cudaFuncSetAttribute(rescore_select_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
      rescore_select_warp_kernel<<<(pp.nq + kRescoreWarps - 1) / kRescoreWarps, 32 * kRescoreWarps, smem, stream>>>(
          q, g, pp.nq, d, k, pp.n_qtiles, pl.n_gtiles, pp.gchunk, pp.n_chunks, pp.n_units, pl.rows_per_qtile, pp.n_sets, pl.d_pad,
          pb.cand, pb.ccnt, pb.cthr, qmap, mu, nu, qflag, qnh, qnr, qnx, gmax, g_index_base,
          g_index_stride, out_scores, out_idx, flagged, n_flagged, thr_next, pp.max_cand);
      count_launch();
      DCR_CUDA_CHECK(cudaGetLastError());
      return 0;
    }
    const size_t rs_smem = ((static_cast<size_t>(d) + 1) & ~size_t(1)) * 8 + static_cast<size_t>(pp.max_cand) * 20 + 16;
    DCR_CUDA_CHECK(cudaFuncSetAttribute(rescore_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(rs_smem)));
    rescore_select_kernel<<<pp.nq, 128, rs_smem, stream>>>(
        q, g, nq, ng, d, k, pp.n_qtiles, pl.n_gtiles, pp.gchunk, pp.n_chunks, pp.n_units, pl.rows_per_qtile, pp.n_sets, pl.d_pad,
        pb.cand, pb.ccnt,
        pb.cthr, qmap, mu, nu, qflag, qnh, qnr, qnx, gmax, g_index_base, g_index_stride, out_scores, out_idx,
        flagged, n_flagged, thr_next, pp.max_cand);
    count_launch();
    DCR_CUDA_CHECK(cudaGetLastError());
    return 0;
  };
  if (int rc = rescore(pl.p0, nullptr, flag0, counts + 0, thr1)) return rc;

  int h_counts[2] = {0, 0};
  unsigned long long h_clk[4] = {0, 0, 0, 0};
  DCR_CUDA_CHECK(cudaMemcpyAsync(h_counts, counts, 8, cudaMemcpyDeviceToHost, stream));
  DCR_CUDA_CHECK(cudaMemcpyAsync(h_clk, clk, 32, cudaMemcpyDeviceToHost, stream));
  DCR_CUDA_CHECK(cudaStreamSynchronize(stream));
  int n_second = 0;
  const int* exact_list = flag0;
  int n_exact = h_counts[0];
  if (h_counts[0] > 0 && pl.kp1) {
    // second chance: the flagged queries alone, 32 candidates per (query, segment)
    n_second = h_counts[0];
    PassPlan p1;
    if (int rc = plan_pass(n_second, pl.kp1, pl, di->num_sms, di->max_smem_optin, d, k, &p1)) return rc;
    gather_rows_kernel<<<std::min(di->num_sms * 8, (p1.nq_pad * (pl.d_pad / 8) + 255) / 256), 256, 0, stream>>>(
        qb, flag0, n_second, p1.nq_pad, pl.d_pad, qb1);
    count_launch();
    if (int rc = launch_fused(pl, p1, qb1, gb, ng, pb, bias, qflag, thr1, nullptr, gthr, stream)) return rc;
    if (int rc = rescore(p1, flag0, flag1, counts + 1, nullptr)) return rc;
    DCR_CUDA_CHECK(cudaMemcpyAsync(h_counts, counts, 8, cudaMemcpyDeviceToHost, stream));
    DCR_CUDA_CHECK(cudaStreamSynchronize(stream));
    exact_list = flag1;
    n_exact = h_counts[1];
  }

  // brute-force fp64 path for the queries whose certificate still fails (ties beyond 32 candidates, NaNs, ...)
  if (n_exact > 0) {
    // queries per brute-force launch: as many as fit in shared memory next to each other (32 up to d = 1536)
    const int ex_batch = std::max(1, std::min<int>(kExactBatch, static_cast<int>(192 * 1024 / (static_cast<size_t>(d) * 4))));
    const size_t ex_smem = static_cast<size_t>(ex_batch) * d * 4;
    DCR_CUDA_CHECK(cudaFuncSetAttribute(exact_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(ex_smem)));
    const int* n_dev = (exact_list == flag0) ? counts + 0 : counts + 1;
    for (int done = 0; done < n_exact; done += ex_batch) {
      exact_scan_kernel<<<di->num_sms * 2, 256, ex_smem, stream>>>(q, g, ng, d, exact_list, done, n_dev, exact, ex_batch);
      count_launch();
      exact_select_kernel<<<ex_batch, 256, 0, stream>>>(exact, ng, k, exact_list, done, n_dev, g_index_base,
                                                           g_index_stride, out_scores, out_idx);
      count_launch();
    }
    DCR_CUDA_CHECK(cudaGetLastError());
    DCR_CUDA_CHECK(cudaStreamSynchronize(stream));
  }

  if (stats) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev0, ev1) != cudaSuccess) ms = 0.f;
    stats->kernel_ms = ms;
    stats->sm_mhz = (h_clk[3] > h_clk[1]) ? static_cast<float>(static_cast<double>(h_clk[2] - h_clk[0]) * 1e3 /
                                                               static_cast<double>(h_clk[3] - h_clk[1]))
                                          : 0.f;
    stats->n_sets = pl.p0.n_sets;
    stats->cta_group = kCG;
    stats->grid = pl.p0.n_units * kCG;
    stats->smem_bytes = static_cast<int>(pl.p0.smem_bytes);
    stats->stages = pl.p0.stages;
    stats->kp = pl.p0.kp;
    stats->cap = pl.p0.cap;
    stats->n_flagged = n_exact;
    stats->n_second = n_second;
    stats->d_pad = pl.d_pad;
  }
  return 0;
}

}  // namespace dcr
