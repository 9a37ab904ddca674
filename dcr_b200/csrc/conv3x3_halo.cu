// 3x3 / stride 1 / pad 1 convolution as an implicit GEMM whose A operand is loaded ONCE per tile.
//
// The generic kernel (conv_gemm.cu) gathers one [128 pixels x 64 channels] A tile per filter tap, i.e. every input
// pixel travels L2 -> shared memory nine times; for the convolutions with few output channels that ingest is the
// bound (DESIGN.md section 5: loads alone took 96 % of the layer time).  Here a tile is R whole output rows of
// one image and the producer loads, per 64-channel block, ONE halo block
//       [(R + 2) input rows] x [(W + 2) pixels, the two extra ones zero-filled by the TMA unit] x [64 channels]
// as a single 4-D tiled TMA box.  In shared memory that is a width-padded raster of 128-byte rows, so the A operand of
// filter tap (r, s) is the SAME buffer read from a start address shifted by (r * (W + 2) + s) rows: nine UMMA descriptor
// start addresses instead of nine loads.  (The 128-byte swizzle is a function of the absolute shared-memory address
// on both the TMA write and the UMMA read side, so a start address that is a multiple of 128 B but not of 1024 B is
// fine.)  MMA row m of the tile is padded-raster position m = pl * (W + 2) + ql; positions with ql >= W (2 per row)
// and the rows past R * (W + 2) are junk that the epilogue drops when it compacts the tile into the [R x W] staging
// box of the TMA store.  W + 2 <= 64 and R = 128 / (W + 2) rows: 2 rows at 56 wide (87.5 % useful MMA rows), 4 at 28,
// 8 at 14.  Used for N <= 128 (measured on B200: 171 -> 89 us at 56x56x64->64, 74 -> 55 us at 28x28x128->128, batch
// 256; at N = 256 only two 32 KB weight stages fit beside the halo buffers and the generic kernel is faster).
//
// Weights are streamed per (tap, channel block) exactly as in the generic kernel (all SMs read the same tiles; that
// traffic is served at several times the rate of per-SM-unique data).  Fast (single-plane bf16) mode only, no residual:
// what the 3x3 convolutions of the ResNet / ResNeXt bottlenecks need.
#include <cuda_bf16.h>

#include <algorithm>
#include <cstring>

#include "dcr_internal.cuh"
#include "host_util.cuh"
#include "ptx.cuh"

namespace dcr {

namespace {

constexpr int kHM = 128;                    // MMA rows (padded-raster positions) per tile
constexpr int kHK = 64;                     // channels per block = one 128-byte swizzled row
constexpr int kSlabBytes = kHM * 128;       // one 64-channel slab of the output staging tile
constexpr int kHThreads = 352;              // warp 0 producer, warp 1 (and 10) MMA issuers, warps 2..9 epilogue

struct HaloMaps {
  CUtensorMap a;     // input  [B][H][W][C]   box 64 x (W+2) x (R+2) x 1
  CUtensorMap w;     // weights [N][9 * cblocks * 64] box 64 x BN
  CUtensorMap out;   // output [B][H][W][ld_out] box 64 x W x R x 1
};

struct HaloParams {
  int H, W, Wp, R, N, cblocks;
  int tiles_per_img, num_tiles;
  int a_bufs, w_stages;
  uint32_t halo_bytes;     // bytes one halo box delivers
  uint32_t a_buf_bytes;    // bytes reserved per halo buffer: the box and the last tap's 128-row window stay inside (1024-aligned)
  const float* scale;
  const float* bias;
  int act, out_col_off;
};

DCR_DEVICE void tma_store_commit_() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
DCR_DEVICE void tma_store_wait_read_() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
DCR_DEVICE void tma_store_wait_all_() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
DCR_DEVICE uint32_t pack_bf16_(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}

// kRW: ALL filter taps stay resident in shared memory (9 * cblocks tiles of [BN x 64]; fits for the 64 -> 64 convolutions of
// ResNet layer1: 72 KB) and TWO warps issue the MMAs, alternating tiles on the two TMEM accumulators.  One thread issues a
// 128 x 64 x 16 tcgen05.mma every ~90 cycles in this loop while the tensor core needs 32 (tools/microbench/umma_rate.cu), and
// with the weight ring gone the two issuers only share the halo buffers, one per tile.
template <int BN, bool kRW>
__global__ void __launch_bounds__(kHThreads, 1)
    conv3x3_halo_kernel(const __grid_constant__ HaloMaps maps, const HaloParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kWStage = BN * 128;
  constexpr uint32_t kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  constexpr int kChunksPerWarp = BN / 64;
  uint8_t* a_ring = smem;
  uint8_t* w_ring = a_ring + p.a_bufs * p.a_buf_bytes;                // kRW: 9 * cblocks resident tiles, tap-major
  uint8_t* out_stage = w_ring + (kRW ? 9 * p.cblocks : p.w_stages) * kWStage;                 // BN/64 slabs
  float* sb = reinterpret_cast<float*>(out_stage + (BN / 64) * kSlabBytes);   // [scale | bias][BN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sb + 2 * BN);
  uint64_t* a_full = bars;          // [4]
  uint64_t* a_empty = bars + 4;     // [4]
  uint64_t* w_full = bars + 8;      // [8]
  uint64_t* w_empty = bars + 16;    // [8]
  uint64_t* t_full = bars + 24;     // [2]
  uint64_t* t_empty = bars + 26;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 28);

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.a);
    tma_prefetch_desc(&maps.w);
    tma_prefetch_desc(&maps.out);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.a_bufs; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < (kRW ? 1 : p.w_stages); ++s) {
      mbar_init(&w_full[s], 1);
      mbar_init(&w_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&t_full[b], 1);
      mbar_init(&t_empty[b], 8);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<1>(tmem_slot, kTmemCols);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    // (whole warp walks the loop, one elected lane issues: see conv_gemm.cu)
    {
      PipeState as(p.a_bufs), ws(kRW ? 1 : p.w_stages);
      if constexpr (kRW) {   // every filter tap once
        if (elect_one()) {
          mbar_arrive_expect_tx(&w_full[0], 9 * p.cblocks * kWStage);
          for (int t = 0; t < 9 * p.cblocks; ++t)
            tma_load_2d<1>(w_ring + t * kWStage, &maps.w, &w_full[0], t * kHK, 0, kEvictLast);
        }
        __syncwarp();
      }
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int b = tile / p.tiles_per_img;
        const int p0 = (tile - b * p.tiles_per_img) * p.R;
        for (int cb = 0; cb < p.cblocks; ++cb, as.next()) {
          const uint32_t sa = as.s, pha = as.ph;
          mbar_wait(&a_empty[sa], pha ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&a_full[sa], p.halo_bytes);
            // rows p0-1 .. p0+R, columns -1 .. W: everything outside the image arrives as zeros (the padding)
            tma_load_4d(a_ring + sa * p.a_buf_bytes, &maps.a, &a_full[sa], cb * kHK, -1, p0 - 1, b, kEvictNormal);
          }
          __syncwarp();
          if constexpr (kRW) continue;
          for (int tap = 0; tap < 9; ++tap, ws.next()) {
            const uint32_t sw = ws.s, phw = ws.ph;
            mbar_wait(&w_empty[sw], phw ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&w_full[sw], kWStage);
              tma_load_2d<1>(w_ring + sw * kWStage, &maps.w, &w_full[sw], (tap * p.cblocks + cb) * kHK, 0, kEvictLast);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp == 1 || (kRW && warp == 10)) {
    // ===================================== MMA issuer(s) =====================================
    {
      constexpr uint32_t idesc = umma_idesc_bf16(kHM, BN);
      const uint32_t issuer = (warp == 1) ? 0u : 1u;
      uint32_t tc = 0;
      PipeState as(p.a_bufs), ws(kRW ? 1 : p.w_stages);
      const uint64_t da0 = umma_desc_sw128(smem_u32(a_ring));
      const uint64_t db0 = umma_desc_sw128(smem_u32(w_ring));
      const uint32_t row_step = static_cast<uint32_t>(p.Wp) * 8u;   // one padded image row in 16-byte units (128 B / pixel)
      if constexpr (kRW) {
        mbar_wait(&w_full[0], 0);
        tc_fence_after();
      }
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tc) {
        const uint32_t buf = tc & 1;
        if (kRW && buf != issuer) {   // the other issuer's tile: only keep the halo ring position in step
          for (int cb = 0; cb < p.cblocks; ++cb) as.next();
          continue;
        }
        mbar_wait(&t_empty[buf], ((tc >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * BN;
        uint32_t accumulate = 0;
        for (int cb = 0; cb < p.cblocks; ++cb, as.next()) {
          const uint32_t sa = as.s;
          mbar_wait(&a_full[sa], as.ph);
          tc_fence_after();
          const uint64_t da_buf = da0 + static_cast<uint64_t>(sa * (p.a_buf_bytes >> 4));
#pragma unroll
          for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int s = 0; s < 3; ++s) {
              uint32_t sw = 0;
              if constexpr (!kRW) {
                sw = ws.s;
                mbar_wait(&w_full[sw], ws.ph);
                tc_fence_after();
              } else {
                sw = static_cast<uint32_t>((r * 3 + s) * p.cblocks + cb);   // resident tile of this (tap, channel block)
              }
              // the tap's view of the halo block: same buffer, start shifted by r padded rows + s pixels (128 B each)
              const uint64_t da = da_buf + static_cast<uint64_t>(r * row_step + s * 8);
              const uint64_t db = db0 + static_cast<uint64_t>(sw * (kWStage >> 4));
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < kHK / 16; ++k) umma_f16<1>(tmem_d, da + 2 * k, db + 2 * k, idesc, accumulate | k);
                if constexpr (!kRW) umma_commit<1>(&w_empty[sw]);
                if (r == 2 && s == 2) {
                  umma_commit<1>(&a_empty[sa]);
                  if (cb == p.cblocks - 1) umma_commit<1>(&t_full[buf]);
                }
              }
              __syncwarp();
              accumulate = 1;
              if constexpr (!kRW) ws.next();
            }
          }
        }
      }
    }
  } else if (warp < 10) {
    // ===================================== epilogue warps =====================================
    const uint32_t ewarp = warp - 2;
    const uint32_t quad = warp & 3;
    const uint32_t half = ewarp >> 2;
    const uint32_t m = quad * 32 + lane;                 // padded-raster position of this thread's accumulator row
    const uint32_t etid = ewarp * 32 + lane;
    const uint32_t tmem_row = tmem_base + ((quad * 32u) << 16);
    const int pl = static_cast<int>(m) / p.Wp, ql = static_cast<int>(m) - pl * p.Wp;
    const bool valid = ql < p.W && pl < p.R;
    const uint32_t srow = static_cast<uint32_t>(pl * p.W + ql);          // row of the compact [R x W] staging box
    const uint32_t sb_addr = smem_u32(sb), stage_addr = smem_u32(out_stage);
    for (int c = etid; c < BN; c += 256) {
      st_shared_f32(sb_addr + c * 4, (p.scale && c < p.N) ? p.scale[c] : 1.f);
      st_shared_f32(sb_addr + (BN + c) * 4, (p.bias && c < p.N) ? p.bias[c] : 0.f);
    }
    uint32_t tc = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tc) {
      const int b = tile / p.tiles_per_img;
      const int p0 = (tile - b * p.tiles_per_img) * p.R;
      const uint32_t buf = tc & 1;
      if (etid == 0) tma_store_wait_read_();     // the previous tile's store has finished reading the staging box
      asm volatile("bar.sync 1, 256;" ::: "memory");   // (also orders the scale/bias staging before its first use)
      mbar_wait(&t_full[buf], (tc >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_row + buf * BN;
#pragma unroll 1
      for (int ci = 0; ci < kChunksPerWarp; ++ci) {
        const int ch = half * kChunksPerWarp + ci;
        uint32_t r[32];
        tmem_ld_32x32(taddr + ch * 32, r);
        tmem_ld_wait_regs(r);
        if (ci == kChunksPerWarp - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&t_empty[buf]);
        }
        if (ch * 32 >= p.N) continue;   // warp-uniform
        float y[32];
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const float4 sc = ld_shared_f4(sb_addr + (ch * 32 + c) * 4);
          const float4 bi = ld_shared_f4(sb_addr + (BN + ch * 32 + c) * 4);
          y[c + 0] = fmaf(__uint_as_float(r[c + 0]), sc.x, bi.x);
          y[c + 1] = fmaf(__uint_as_float(r[c + 1]), sc.y, bi.y);
          y[c + 2] = fmaf(__uint_as_float(r[c + 2]), sc.z, bi.z);
          y[c + 3] = fmaf(__uint_as_float(r[c + 3]), sc.w, bi.w);
        }
        if (p.act == 1) {
#pragma unroll
          for (int c = 0; c < 32; ++c) y[c] = fmaxf(y[c], 0.f);
        }
        const uint32_t dst = stage_addr + (ch >> 1) * kSlabBytes + srow * 128;
        const uint32_t sw = srow & 7;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 v;
          v.x = pack_bf16_(y[j * 8 + 0], y[j * 8 + 1]);
          v.y = pack_bf16_(y[j * 8 + 2], y[j * 8 + 3]);
          v.z = pack_bf16_(y[j * 8 + 4], y[j * 8 + 5]);
          v.w = pack_bf16_(y[j * 8 + 6], y[j * 8 + 7]);
          if (valid) st_shared_v4(dst + ((((ch & 1) * 4 + j) ^ sw) << 4), v);   // junk positions are dropped here
        }
        __syncwarp();
      }
      fence_proxy_async();
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (etid == 0) {
        for (int sl = 0; sl < BN / 64; ++sl)
          if (sl * 64 < p.N) tma_store_4d(&maps.out, out_stage + sl * kSlabBytes, p.out_col_off + sl * 64, 0, p0, b);
        tma_store_commit_();
      }
    }
    if (etid == 0) tma_store_wait_all_();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<1>(tmem_base, kTmemCols);
}

template <int BN, bool kRW>
int launch_halo(const HaloMaps& maps, HaloParams& p, int num_sms, size_t max_smem, cudaStream_t stream) {
  constexpr size_t kWStage = static_cast<size_t>(BN) * 128;
  const size_t fixed = 1024 + static_cast<size_t>(BN / 64) * kSlabBytes + 2 * BN * 4 + 256;
  const size_t abuf = p.a_buf_bytes;
  size_t smem = 0;
  if constexpr (kRW) {
    const size_t wres = static_cast<size_t>(9) * p.cblocks * kWStage;
    DCR_REQUIRE(max_smem >= fixed + wres + 2 * abuf, "conv3x3_halo: resident weights do not fit");
    p.a_bufs = static_cast<int>(std::min<size_t>(4, (max_smem - fixed - wres) / abuf));
    p.w_stages = 0;
    smem = fixed + wres + static_cast<size_t>(p.a_bufs) * abuf;
  } else {
    // two halo buffers and 3..8 weight stages; a third halo buffer if 6 weight stages still fit beside it
    p.a_bufs = 2;
    DCR_REQUIRE(max_smem >= fixed + 2 * abuf + 3 * kWStage, "conv3x3_halo: not enough shared memory");
    p.w_stages = static_cast<int>(std::min<size_t>(8, (max_smem - fixed - 2 * abuf) / kWStage));
    if (max_smem >= fixed + 3 * abuf + 6 * kWStage) {
      p.a_bufs = 3;
      p.w_stages = static_cast<int>(std::min<size_t>(8, (max_smem - fixed - 3 * abuf) / kWStage));
    }
    smem = fixed + static_cast<size_t>(p.a_bufs) * abuf + static_cast<size_t>(p.w_stages) * kWStage;
  }
  auto kern = conv3x3_halo_kernel<BN, kRW>;
  static bool attr_set_dev[64] = {};   // per template instantiation and device (the attribute is per device)
  int cur_dev = 0;
  DCR_CUDA_CHECK(cudaGetDevice(&cur_dev));
  bool& attr_set = attr_set_dev[cur_dev & 63];
  if (!attr_set) {
    DCR_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(max_smem)));
    attr_set = true;
  }
  kern<<<std::min(p.num_tiles, num_sms), kHThreads, smem, stream>>>(maps, p);
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

bool conv3x3_halo_eligible(const ConvGemmDesc& d) {
  if (tuning_flag("DCR_CONV_NO_HALO")) return false;
  const bool shape = d.kh == 3 && d.kw == 3 && d.stride == 1 && d.pad_h == 1 && d.pad_w == 1 && d.in_stride_w == 0;
  const bool fast = d.n_terms == 1 && d.term_a[0] == 0 && d.term_w[0] == 0 && !d.exact && d.out != nullptr &&
                    d.out_planes <= 1 && d.out_f32 == nullptr && d.res == nullptr && (d.act == 0 || d.act == 1);
  const bool dims = d.C % 64 == 0 && d.ld_in == d.C && d.N % 64 == 0 && d.N <= 128 && d.ld_out % 8 == 0 &&
                    d.out_col_off % 8 == 0 && d.W + 2 <= 64 && d.W >= 8 && d.H >= 2 && d.B >= 1;
  return shape && fast && dims;
}

int conv3x3_halo(const ConvGemmDesc& d, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  HaloParams p;
  memset(&p, 0, sizeof(p));
  p.H = d.H; p.W = d.W; p.Wp = d.W + 2;
  p.R = std::min(kHM / p.Wp, d.H);
  p.N = d.N;
  p.cblocks = d.C / 64;
  p.tiles_per_img = (d.H + p.R - 1) / p.R;
  p.num_tiles = d.B * p.tiles_per_img;
  p.halo_bytes = static_cast<uint32_t>(128) * p.Wp * (p.R + 2);
  p.scale = d.scale; p.bias = d.bias; p.act = d.act; p.out_col_off = d.out_col_off;
  // the loaded block and the last tap's 128-row window (start row 2 * Wp + 2) must stay inside the buffer
  p.a_buf_bytes = (std::max<uint32_t>(p.halo_bytes, static_cast<uint32_t>(2 * p.Wp + 2 + kHM) * 128u) + 1023u) & ~1023u;
  HaloMaps maps;
  memset(&maps, 0, sizeof(maps));
  if (int rc = make_tmap_nhwc_box_bf16(&maps.a, d.in, d.B, d.H, d.W, d.C, d.C, p.Wp, p.R + 2)) return rc;
  const int BN = d.N <= 64 ? 64 : 128;   // conv3x3_halo_eligible: N is 64 or 128
  const int ktot = 9 * p.cblocks * 64;
  if (int rc = make_tmap_2d_bf16(&maps.w, d.weight, d.N, ktot, ktot, BN, 64)) return rc;
  if (int rc = make_tmap_nhwc_box_bf16(&maps.out, d.out, d.B, d.H, d.W, d.ld_out, d.ld_out, d.W, p.R)) return rc;
  // all taps resident + two MMA issuers when the weights are small (ResNet layer1: 9 x [64 x 64] = 72 KB)
  const bool resident = BN == 64 && static_cast<size_t>(9) * p.cblocks * BN * 128 <= 80 * 1024;
  if (BN == 64) return resident ? launch_halo<64, true>(maps, p, di->num_sms, di->max_smem_optin, stream)
                                : launch_halo<64, false>(maps, p, di->num_sms, di->max_smem_optin, stream);
  return launch_halo<128, false>(maps, p, di->num_sms, di->max_smem_optin, stream);
}

}  // namespace dcr
