// Cross-layer fusion of the ResNet bottleneck's 1x1 pair (sm_100a, tcgen05 + TMA):
//
//     Y  = relu(scale3 * (T2 @ W3^T) + bias3 + X)        conv3 (1x1 expand) + BN + residual + ReLU of block i
//     T1 = relu(scale1 * (Y  @ W1^T) + bias1)            conv1 (1x1 reduce) + BN + ReLU of block i+1
//
// as ONE kernel.  Unfused, the expanded activation Y (B*H*W x 4*width bf16: 411 MB at 56x56, batch 256) is written by the
// first GEMM and read again by the second -- and both GEMMs already run at the HBM roofline (profiles/r01_layers_sscd.txt:
// 5.9 / 6.5 TB/s of algorithmic bytes).  Here a CTA keeps the 128 rows of T2 it works on resident, walks the column
// blocks of Y, and every finished 128x128 block of Y is (a) stored to HBM (block i+1 still needs it as its residual) and
// (b) consumed IN PLACE from the store's 128B-swizzled staging tile as the A operand of the second GEMM, whose
// accumulator lives in its own TMEM columns.  Y is never read back: per row 2*(K1 + 2*N1 + N2) bytes instead of
// 2*(K1 + 3*N1 + N2) -- 1028 instead of 1439 MB per layer1 block pair.
//
// Reference call sites replaced (through `model(samples)`, utils_ret.py:751): torchvision Bottleneck.forward's
// conv3/bn3/+identity/relu of one block and conv1/bn1/relu of the next (SSCD trunk, SURVEY.md 8a4).
//
// Roles (320 threads, persistent over 128-row m-tiles):  warp 0 TMA producer, warp 1 tcgen05.mma issuer, warps 2-9 epilogue.
//   shared memory   A1 (T2 rows, all of K1; 1-2 buffers) | W ring (16 KB stages: W3 tiles and W1 slabs in issue order) |
//                   3 rotating X tiles (128 x 128 bf16: residual lands here by TMA, the epilogue overwrites it in place
//                   with Y, the TMA store and the second GEMM read it) | T1 staging | BN tables | mbarriers
//   tensor memory   [0,256) two accumulators of the first GEMM, [256, 256+N2) accumulator of the second
// Results are bit-identical to the two separate launches of conv_gemm.cu (same K order, same epilogue arithmetic).
#include <cuda_bf16.h>

#include <algorithm>
#include <cstring>

#include "dcr_internal.cuh"
#include "host_util.cuh"
#include "ptx.cuh"

namespace dcr {

namespace {

constexpr int kFM = 128;                 // rows per m-tile (TMEM lanes)
constexpr int kFN = 128;                 // columns of Y per n-block
constexpr int kFK = 64;                  // bf16 per 128-byte swizzled row
constexpr int kFThreads = 320;
constexpr int kSlab = kFM * 128;         // one [128 rows x 64 bf16] slab, 16 KB
constexpr int kXTile = 2 * kSlab;        // one 128 x 128 tile of X / Y
constexpr int kXBufs = 3;
constexpr int kWStage = kSlab;           // 16 KB: a W3 tile [128 x 64] or a W1 slab [N2 <= 128 x 64]
constexpr uint32_t kAcc2Col = 256;       // TMEM column of the second accumulator

struct FuseMaps {
  CUtensorMap a;      // T2   [M, K1]   box 128 x 64
  CUtensorMap w3;     // W3   [N1, K1]  box 128 x 64
  CUtensorMap res;    // X    [M, N1]   box 128 x 64
  CUtensorMap out;    // Y    [M, N1]   box 128 x 64
  CUtensorMap w1;     // W1   [N2, N1]  box N2 x 64
  CUtensorMap out2;   // T1   [M, N2]   box 128 x 64
};

struct FuseParams {
  int M, N1, N2;
  int k_iters1;       // K1 / 64
  int nb;             // N1 / 128
  int num_m_tiles;
  int a_bufs, w_stages;
  const float* scale3;
  const float* bias3;
  const float* scale1;
  const float* bias1;
};

DCR_DEVICE uint32_t pack2(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}
DCR_DEVICE void store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
DCR_DEVICE void store_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
DCR_DEVICE void store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
DCR_DEVICE void tma_store_2d_(const void* tmap, uint32_t src_smem, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}

// N2 = 0: expansion only (no following reduce convolution to fuse with) -- the same in-place residual / three rotating
// tile pipeline for the 1x1 expansions whose separate staging tiles do not fit beside the resident A rows in conv_gemm.cu
// (K = 256: layer3 of the ResNet-50, where that kernel has to serialise on a single output staging tile).
template <int N2>
__global__ void __launch_bounds__(kFThreads, 1) expand_reduce_kernel(const __grid_constant__ FuseMaps maps, const FuseParams p) {
  static_assert(N2 == 0 || N2 == 64 || N2 == 128, "second GEMM width");
  constexpr bool kSecond = N2 != 0;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int k_iters1 = p.k_iters1, nb = p.nb;
  const int a_buf_bytes = k_iters1 * kSlab;
  uint8_t* smem_a = smem;                                           // a_bufs x k_iters1 slabs
  uint8_t* smem_w = smem_a + p.a_bufs * a_buf_bytes;                // w_stages x 16 KB
  uint8_t* smem_x = smem_w + p.w_stages * kWStage;                  // 3 x 32 KB
  uint8_t* smem_o2 = smem_x + kXBufs * kXTile;                      // N2/64 slabs
  float* sb = reinterpret_cast<float*>(smem_o2 + (N2 / 64) * kSlab);   // scale3[N1] | bias3[N1] | scale1[N2] | bias1[N2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sb + 2 * p.N1 + 2 * N2);
  uint64_t* a_full = bars;            // [2]
  uint64_t* a_empty = bars + 2;       // [2]
  uint64_t* w_full = bars + 4;        // [8]
  uint64_t* w_empty = bars + 12;      // [8]
  uint64_t* t_full = bars + 20;       // [2]
  uint64_t* t_empty = bars + 22;      // [2]
  uint64_t* r_full = bars + 24;       // [3] residual tile landed in X buffer b
  uint64_t* y_ready = bars + 27;      // [3] epilogue finished writing Y into X buffer b
  uint64_t* y_free = bars + 30;       // [3] second GEMM finished reading X buffer b
  uint64_t* acc2_full = bars + 33;
  uint64_t* acc2_empty = bars + 34;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 35);

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.a);
    tma_prefetch_desc(&maps.w3);
    tma_prefetch_desc(&maps.res);
    tma_prefetch_desc(&maps.out);
    tma_prefetch_desc(&maps.w1);
    tma_prefetch_desc(&maps.out2);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
      mbar_init(&t_full[s], 1);
      mbar_init(&t_empty[s], 8);
    }
    for (int s = 0; s < 8; ++s) {
      mbar_init(&w_full[s], 1);
      mbar_init(&w_empty[s], 1);
    }
    for (int s = 0; s < kXBufs; ++s) {
      mbar_init(&r_full[s], 1);
      mbar_init(&y_ready[s], 1);
      mbar_init(&y_free[s], 1);
    }
    mbar_init(acc2_full, 1);
    mbar_init(acc2_empty, 8);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_m_tiles = p.num_m_tiles;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    PipeState ws(p.w_stages), as(p.a_bufs);
    for (int tile = blockIdx.x; tile < num_m_tiles; tile += gridDim.x, as.next()) {
      const int m0 = tile * kFM;
      mbar_wait(&a_empty[as.s], as.ph ^ 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(&a_full[as.s], a_buf_bytes);
        for (int ki = 0; ki < k_iters1; ++ki)
          tma_load_2d<1>(smem_a + as.s * a_buf_bytes + ki * kSlab, &maps.a, &a_full[as.s], ki * kFK, m0, kEvictFirst);
      }
      __syncwarp();
      for (int j = 0; j <= nb; ++j) {
        if (j < nb) {   // W3 tiles of column block j
          for (int ki = 0; ki < k_iters1; ++ki, ws.next()) {
            mbar_wait(&w_empty[ws.s], ws.ph ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&w_full[ws.s], kFN * 128);
              tma_load_2d<1>(smem_w + ws.s * kWStage, &maps.w3, &w_full[ws.s], ki * kFK, j * kFN, kEvictLast);
            }
            __syncwarp();
          }
        }
        if (kSecond && j >= 1) {   // W1 slabs matching the two 64-column slabs of Y block j-1
          for (int sl = 0; sl < 2; ++sl, ws.next()) {
            mbar_wait(&w_empty[ws.s], ws.ph ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&w_full[ws.s], N2 * 128);
              tma_load_2d<1>(smem_w + ws.s * kWStage, &maps.w1, &w_full[ws.s], ((j - 1) * 2 + sl) * kFK, 0, kEvictLast);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =====================================
    constexpr uint32_t idesc1 = umma_idesc_bf16(kFM, kFN);
    constexpr uint32_t idesc2 = umma_idesc_bf16(kFM, kSecond ? N2 : 64);
    PipeState ws(p.w_stages), as(p.a_bufs), xs(kXBufs);
    const uint64_t da0 = umma_desc_sw128(smem_u32(smem_a));
    const uint64_t dw0 = umma_desc_sw128(smem_u32(smem_w));
    const uint64_t dx0 = umma_desc_sw128(smem_u32(smem_x));
    const uint32_t tmem_acc2 = tmem_base + kAcc2Col;
    uint32_t g = 0, mt = 0;
    for (int tile = blockIdx.x; tile < num_m_tiles; tile += gridDim.x, ++mt, as.next()) {
      mbar_wait(&a_full[as.s], as.ph);
      tc_fence_after();
      const uint64_t da_buf = da0 + static_cast<uint64_t>(as.s * (a_buf_bytes >> 4));
      for (int j = 0; j <= nb; ++j) {
        if (j < nb) {   // first GEMM, column block j -> accumulator g & 1
          const uint32_t buf = g & 1;
          mbar_wait(&t_empty[buf], ((g >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + buf * kFN;
          for (int ki = 0; ki < k_iters1; ++ki, ws.next()) {
            mbar_wait(&w_full[ws.s], ws.ph);
            tc_fence_after();
            const uint64_t da = da_buf + static_cast<uint64_t>(ki * (kSlab >> 4));
            const uint64_t db = dw0 + static_cast<uint64_t>(ws.s * (kWStage >> 4));
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < kFK / 16; ++k) umma_f16<1>(tmem_d, da + 2 * k, db + 2 * k, idesc1, (ki | k) != 0);
              umma_commit<1>(&w_empty[ws.s]);
              if (ki == k_iters1 - 1) {
                umma_commit<1>(&t_full[buf]);
                if (j == nb - 1) umma_commit<1>(&a_empty[as.s]);
              }
            }
            __syncwarp();
          }
          ++g;
        }
        if (kSecond && j >= 1) {   // second GEMM: acc2 += Y block j-1 (in X buffer xs.s) x W1 slabs
          mbar_wait(&y_ready[xs.s], xs.ph);
          if (j == 1) mbar_wait(acc2_empty, (mt & 1) ^ 1);   // previous m-tile's T1 epilogue has drained acc2
          tc_fence_after();
          for (int sl = 0; sl < 2; ++sl, ws.next()) {
            mbar_wait(&w_full[ws.s], ws.ph);
            tc_fence_after();
            const uint64_t da = dx0 + static_cast<uint64_t>(xs.s * (kXTile >> 4) + sl * (kSlab >> 4));
            const uint64_t db = dw0 + static_cast<uint64_t>(ws.s * (kWStage >> 4));
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < kFK / 16; ++k) umma_f16<1>(tmem_acc2, da + 2 * k, db + 2 * k, idesc2, (j > 1) || (sl | k) != 0);
              umma_commit<1>(&w_empty[ws.s]);
              if (sl == 1) {
                umma_commit<1>(&y_free[xs.s]);
                if (j == nb) umma_commit<1>(acc2_full);
              }
            }
            __syncwarp();
          }
          xs.next();
        }
      }
    }
  } else {
    // ===================================== epilogue warps =====================================
    const uint32_t ewarp = warp - 2;               // 0..7
    const uint32_t quad = warp & 3;                // TMEM lane quadrant
    const uint32_t half = ewarp >> 2;              // which 64-column slab of a 128-column tile
    const uint32_t row = quad * 32 + lane;
    const uint32_t etid = ewarp * 32 + lane;
    const uint32_t tmem_row = tmem_base + ((quad * 32u) << 16);
    const uint32_t sb_addr = smem_u32(sb), x_addr = smem_u32(smem_x), o2_addr = smem_u32(smem_o2);
    const int N1 = p.N1;
    for (int c = etid; c < N1; c += 256) {
      st_shared_f32(sb_addr + c * 4, p.scale3 ? p.scale3[c] : 1.f);
      st_shared_f32(sb_addr + (N1 + c) * 4, p.bias3 ? p.bias3[c] : 0.f);
    }
    for (int c = etid; c < N2; c += 256) {
      st_shared_f32(sb_addr + (2 * N1 + c) * 4, p.scale1 ? p.scale1[c] : 1.f);
      st_shared_f32(sb_addr + (2 * N1 + N2 + c) * 4, p.bias1 ? p.bias1[c] : 0.f);
    }
    // residual of the very first tile
    if (etid == 0 && static_cast<int>(blockIdx.x) < num_m_tiles) {
      mbar_arrive_expect_tx(&r_full[0], kXTile);
      for (int sl = 0; sl < 2; ++sl)
        tma_load_2d<1>(smem_x + sl * kSlab, &maps.res, &r_full[0], sl * kFK, blockIdx.x * kFM, kEvictFirst);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    PipeState xs(kXBufs);
    uint32_t g = 0, mt = 0;
    const uint32_t sw = row & 7;
    for (int tile = blockIdx.x; tile < num_m_tiles; tile += gridDim.x, ++mt) {
      const int m0 = tile * kFM;
      for (int j = 0; j < nb; ++j, ++g, xs.next()) {
        const uint32_t buf = g & 1;
        const uint32_t xb = xs.s;
        if (etid == 0) {
          // prefetch the residual of the NEXT n-tile (possibly the first of this CTA's next m-tile) into the buffer
          // tile g-2 used: its TMA store must have finished reading it and the second GEMM must have consumed it
          const bool has_next = (j + 1 < nb) || (tile + static_cast<int>(gridDim.x) < num_m_tiles);
          if (has_next) {
            const uint32_t xn = (xb + 1 == kXBufs) ? 0 : xb + 1;
            if (g >= 2) {
              store_wait_read_1();
              if constexpr (kSecond) {
                const uint32_t ph_prev = (xb >= 2) ? xs.ph : (xs.ph ^ 1);   // parity of use (g-2)/3 of buffer xn
                mbar_wait(&y_free[xn], ph_prev);
              }
            }
            const int nm0 = (j + 1 < nb) ? m0 : (tile + static_cast<int>(gridDim.x)) * kFM;
            const int nn0 = (j + 1 < nb) ? (j + 1) * kFN : 0;
            mbar_arrive_expect_tx(&r_full[xn], kXTile);
            for (int sl = 0; sl < 2; ++sl)
              tma_load_2d<1>(smem_x + xn * kXTile + sl * kSlab, &maps.res, &r_full[xn], nn0 + sl * kFK, nm0, kEvictFirst);
          }
        }
        mbar_wait(&t_full[buf], (g >> 1) & 1);
        tc_fence_after();
        mbar_wait(&r_full[xb], xs.ph);
        const uint32_t taddr = tmem_row + buf * kFN + half * 64;
        const uint32_t xrow = x_addr + xb * kXTile + half * kSlab + row * 128;
        const uint32_t s_scale = sb_addr + (j * kFN + half * 64) * 4;
        const uint32_t s_bias = s_scale + N1 * 4;
#pragma unroll 1
        for (int ci = 0; ci < 2; ++ci) {
          uint32_t r[32];
          tmem_ld_32x32(taddr + ci * 32, r);
          tmem_ld_wait_regs(r);
          if (ci == 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&t_empty[buf]);
          }
          float y[32];
#pragma unroll
          for (int c = 0; c < 32; c += 4) {
            const float4 sc = ld_shared_f4(s_scale + (ci * 32 + c) * 4);
            const float4 bi = ld_shared_f4(s_bias + (ci * 32 + c) * 4);
            y[c + 0] = fmaf(__uint_as_float(r[c + 0]), sc.x, bi.x);
            y[c + 1] = fmaf(__uint_as_float(r[c + 1]), sc.y, bi.y);
            y[c + 2] = fmaf(__uint_as_float(r[c + 2]), sc.z, bi.z);
            y[c + 3] = fmaf(__uint_as_float(r[c + 3]), sc.w, bi.w);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {   // residual: this thread's 16-byte chunks of its row, read then overwritten in place
            const uint32_t addr = xrow + (((ci * 4 + q) ^ sw) << 4);
            const uint4 rv = ld_shared_v4(addr);
            const uint32_t w[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              y[q * 8 + 2 * e] += __uint_as_float(w[e] << 16);
              y[q * 8 + 2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u);
            }
            uint4 v;
            v.x = pack2(fmaxf(y[q * 8 + 0], 0.f), fmaxf(y[q * 8 + 1], 0.f));
            v.y = pack2(fmaxf(y[q * 8 + 2], 0.f), fmaxf(y[q * 8 + 3], 0.f));
            v.z = pack2(fmaxf(y[q * 8 + 4], 0.f), fmaxf(y[q * 8 + 5], 0.f));
            v.w = pack2(fmaxf(y[q * 8 + 6], 0.f), fmaxf(y[q * 8 + 7], 0.f));
            st_shared_v4(addr, v);
          }
        }
        fence_proxy_async();   // generic-proxy writes -> visible to the TMA store and to tcgen05.mma (async proxy)
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (etid == 0) {
          for (int sl = 0; sl < 2; ++sl)
            tma_store_2d_(&maps.out, x_addr + xb * kXTile + sl * kSlab, j * kFN + sl * kFK, m0);
          store_commit();
          if constexpr (kSecond) mbar_arrive(&y_ready[xb]);
        }
      }
      if constexpr (!kSecond) continue;
      // ---- T1 tile of this m-tile: acc2 -> BN + ReLU -> bf16 -> staging -> TMA store ----
      if (etid == 0) store_wait_read_1();   // the previous m-tile's T1 store has finished reading the staging slabs
      asm volatile("bar.sync 1, 256;" ::: "memory");
      mbar_wait(acc2_full, mt & 1);
      tc_fence_after();
      {
        constexpr int kCh = N2 / 64;   // 32-column chunks per warp
        const uint32_t s_scale2 = sb_addr + 2 * N1 * 4;
        const uint32_t s_bias2 = s_scale2 + N2 * 4;
#pragma unroll 1
        for (int ci = 0; ci < kCh; ++ci) {
          const int ch = half * kCh + ci;
          uint32_t r[32];
          tmem_ld_32x32(tmem_row + kAcc2Col + ch * 32, r);
          tmem_ld_wait_regs(r);
          if (ci == kCh - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc2_empty);
          }
          float y[32];
#pragma unroll
          for (int c = 0; c < 32; c += 4) {
            const float4 sc = ld_shared_f4(s_scale2 + (ch * 32 + c) * 4);
            const float4 bi = ld_shared_f4(s_bias2 + (ch * 32 + c) * 4);
            y[c + 0] = fmaxf(fmaf(__uint_as_float(r[c + 0]), sc.x, bi.x), 0.f);
            y[c + 1] = fmaxf(fmaf(__uint_as_float(r[c + 1]), sc.y, bi.y), 0.f);
            y[c + 2] = fmaxf(fmaf(__uint_as_float(r[c + 2]), sc.z, bi.z), 0.f);
            y[c + 3] = fmaxf(fmaf(__uint_as_float(r[c + 3]), sc.w, bi.w), 0.f);
          }
          const uint32_t orow = o2_addr + (ch >> 1) * kSlab + row * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 v;
            v.x = pack2(y[q * 8 + 0], y[q * 8 + 1]);
            v.y = pack2(y[q * 8 + 2], y[q * 8 + 3]);
            v.z = pack2(y[q * 8 + 4], y[q * 8 + 5]);
            v.w = pack2(y[q * 8 + 6], y[q * 8 + 7]);
            st_shared_v4(orow + ((((ch & 1) * 4 + q) ^ sw) << 4), v);
          }
        }
      }
      fence_proxy_async();
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (etid == 0) {
        for (int sl = 0; sl < N2 / 64; ++sl) tma_store_2d_(&maps.out2, o2_addr + sl * kSlab, sl * kFK, m0);
        store_commit();
      }
    }
    if (etid == 0) store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, 512);
}

}  // namespace

bool expand_only_eligible(const ConvGemmDesc& a, size_t max_smem) {
  if (tuning_flag("DCR_NO_BLOCK_FUSION")) return false;
  const bool plain = a.kh == 1 && a.kw == 1 && a.stride == 1 && a.pad_h == 0 && a.pad_w == 0 && a.in_stride_w == 0 && a.n_terms == 1 &&
                     a.term_a[0] == 0 && a.term_w[0] == 0 && !a.exact && a.out != nullptr && a.out_planes <= 1 && a.out_f32 == nullptr &&
                     a.out_col_off == 0 && a.act == 1;
  if (!plain || a.res == nullptr || a.res_planes > 1) return false;
  // K = 64 / 128 expansions keep double-buffered staging in conv_gemm.cu and run at the HBM roofline there already
  if (a.C != 256 || a.ld_in != a.C || a.N % 128 != 0 || a.N > 2048 || a.ld_out != a.N || a.ld_res != a.N) return false;
  const size_t need = 1024 + static_cast<size_t>(a.C / 64) * kSlab + 3 * kWStage + kXBufs * kXTile + 2 * a.N * 4 + 512;
  return need <= max_smem;
}

bool expand_reduce_eligible(const ConvGemmDesc& a, const ConvGemmDesc& b, size_t max_smem) {
  if (tuning_flag("DCR_NO_BLOCK_FUSION")) return false;
  auto plain = [](const ConvGemmDesc& d) {
    return d.kh == 1 && d.kw == 1 && d.stride == 1 && d.pad_h == 0 && d.pad_w == 0 && d.in_stride_w == 0 && d.n_terms == 1 &&
           d.term_a[0] == 0 && d.term_w[0] == 0 && !d.exact && d.out != nullptr && d.out_planes <= 1 && d.out_f32 == nullptr &&
           d.out_col_off == 0 && d.act == 1;
  };
  if (!plain(a) || !plain(b)) return false;
  if (a.res == nullptr || a.res_planes > 1 || b.res != nullptr) return false;
  if (b.in != a.out || b.C != a.N || b.B != a.B || b.H != a.H || b.W != a.W || b.ld_in != a.ld_out) return false;
  if (a.C % 64 != 0 || a.C > 256 || a.ld_in != a.C) return false;
  if (a.N % 128 != 0 || a.ld_out != a.N || a.ld_res != a.N) return false;
  if (!(b.N == 64 || b.N == 128) || b.ld_out != b.N) return false;
  const size_t need = 1024 + static_cast<size_t>(a.C / 64) * kSlab + 3 * kWStage + kXBufs * kXTile + static_cast<size_t>(b.N / 64) * kSlab +
                      (2 * a.N + 2 * b.N) * 4 + 512;
  return need <= max_smem;
}

namespace {
template <int N2>
int launch_fused(const FuseMaps& maps, const FuseParams& p, int grid, size_t smem, const DeviceInfo* di, cudaStream_t stream) {
  static bool attr_set[64] = {};
  if (!attr_set[di->device & 63]) {
    DCR_CUDA_CHECK(cudaFuncSetAttribute(expand_reduce_kernel<N2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(di->max_smem_optin)));
    attr_set[di->device & 63] = true;
  }
  expand_reduce_kernel<N2><<<grid, kFThreads, smem, stream>>>(maps, p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}
}  // namespace

// b == nullptr: expansion only
static int expand_reduce_impl(const ConvGemmDesc& a, const ConvGemmDesc* b, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(di->cc_major == 10, "expand_reduce: this build targets sm_100a; device reports sm_%d%d", di->cc_major, di->cc_minor);
  const long long M = static_cast<long long>(a.B) * a.H * a.W;
  DCR_REQUIRE(M > 0 && M < (1ll << 31), "expand_reduce: M out of range");
  const int n2 = b ? b->N : 0;
  FuseMaps maps;
  memset(&maps, 0, sizeof(maps));
  if (int rc = make_tmap_2d_bf16(&maps.a, a.in, M, a.C, a.ld_in, kFM, kFK)) return rc;
  if (int rc = make_tmap_2d_bf16(&maps.w3, a.weight, a.N, a.C, a.C, kFN, kFK)) return rc;
  if (int rc = make_tmap_2d_bf16(&maps.res, a.res, M, a.N, a.ld_res, kFM, kFK)) return rc;
  if (int rc = make_tmap_2d_bf16(&maps.out, a.out, M, a.N, a.ld_out, kFM, kFK)) return rc;
  if (b) {
    if (int rc = make_tmap_2d_bf16(&maps.w1, b->weight, b->N, b->C, b->C, b->N, kFK)) return rc;
    if (int rc = make_tmap_2d_bf16(&maps.out2, b->out, M, b->N, b->ld_out, kFM, kFK)) return rc;
  } else {
    maps.w1 = maps.w3;
    maps.out2 = maps.out;
  }
  FuseParams p;
  memset(&p, 0, sizeof(p));
  p.M = static_cast<int>(M);
  p.N1 = a.N;
  p.N2 = n2;
  p.k_iters1 = a.C / 64;
  p.nb = a.N / kFN;
  p.num_m_tiles = static_cast<int>((M + kFM - 1) / kFM);
  p.scale3 = a.scale; p.bias3 = a.bias;
  p.scale1 = b ? b->scale : nullptr; p.bias1 = b ? b->bias : nullptr;
  const size_t fixed = 1024 + kXBufs * kXTile + static_cast<size_t>(n2 / 64) * kSlab + (2 * a.N + 2 * n2) * 4 + 512;
  const size_t a_buf = static_cast<size_t>(p.k_iters1) * kSlab;
  // a second buffer for the resident T2 rows when four W stages still fit beside it
  p.a_bufs = (fixed + 2 * a_buf + 4 * kWStage <= di->max_smem_optin) ? 2 : 1;
  p.w_stages = static_cast<int>(std::min<size_t>(8, (di->max_smem_optin - fixed - p.a_bufs * a_buf) / kWStage));
  DCR_REQUIRE(p.w_stages >= 3, "expand_reduce: not enough shared memory");
  const size_t smem = fixed + p.a_bufs * a_buf + static_cast<size_t>(p.w_stages) * kWStage;
  const int grid = std::min(p.num_m_tiles, di->num_sms);
  if (n2 == 0) return launch_fused<0>(maps, p, grid, smem, di, stream);
  if (n2 == 64) return launch_fused<64>(maps, p, grid, smem, di, stream);
  return launch_fused<128>(maps, p, grid, smem, di, stream);
}

int expand_reduce(const ConvGemmDesc& a, const ConvGemmDesc& b, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(expand_reduce_eligible(a, b, di->max_smem_optin), "expand_reduce: layer pair not eligible for fusion");
  return expand_reduce_impl(a, &b, stream);
}

int expand_only(const ConvGemmDesc& a, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(expand_only_eligible(a, di->max_smem_optin), "expand_only: layer not eligible");
  return expand_reduce_impl(a, nullptr, stream);
}

}  // namespace dcr
