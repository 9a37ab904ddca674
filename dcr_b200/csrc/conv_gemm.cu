// tcgen05 GEMM / implicit-GEMM convolution with fused epilogue (sm_100a).
//
// One kernel family computes   Y[m, n] = act( scale[n] * sum_k A[m, k] * W[n, k] + bias[n] (+ R[m, n]) )
// for every dense contraction of the descriptor networks:
//   - 1x1 stride-1 convolutions and Linear layers: A is the NHWC activation matrix [M = B*H*W, K = C]   (TILED)
//   - kxk / strided convolutions: A rows are gathered on the fly by TMA im2col loads from the NHWC tensor,
//     one (filter tap, 64-channel block) per pipeline stage -- the im2col matrix never exists in HBM   (IM2COL)
// Reference call sites this replaces (all reached through `model(samples)`, utils_ret.py:751):
//   SSCD ResNet-50 trunk convs + BN + ReLU (+ residual)            (torchvision resnet50; SURVEY.md 8a4)
//   DINO ViT-S qkv / proj / fc1(+GELU) / fc2 Linear layers          dino_vits.py:96-102,119,127
//   FID Inception BasicConv2d (conv + BN eps=1e-3 + ReLU)           metrics/inception.py:197-341
//
// Precision: operands are bf16 "planes".  Fast mode uses one plane (plain bf16 x bf16 -> fp32).  Parity mode
// stores every activation / weight as 2-3 bf16 planes (hi, mid, lo with x = hi + mid + lo to ~2^-24) and
// accumulates the listed cross terms into the same TMEM accumulator, which reproduces fp32 arithmetic on the
// tensor cores (DESIGN.md section 5).
//
// Structure per CTA (192 threads, persistent over output tiles of 128 x BN):
//   warp 0 : TMA producer (A tile 128x64, W tile BNx64 per stage, 128B swizzle)
//   warp 1 : tcgen05.mma issuer (cta_group::1, UMMA 128 x BN x 16), accumulators double-buffered in TMEM
//   warps 2-5 : epilogue (tcgen05.ld -> scale/bias/residual/activation -> bf16 planes / fp32 -> global)
#include <cuda_bf16.h>

#include <algorithm>
#include <cstring>

#include "dcr_internal.cuh"
#include "host_util.cuh"
#include "ptx.cuh"

namespace dcr {

namespace {

constexpr int kBM = 128;
constexpr int kBK = 64;
constexpr int kThreads = 320;   // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue
constexpr int kAStage = kBM * kBK * 2;   // 16 KB
// direct epilogue: per epilogue warp a [32 rows][64 B + 16 B pad] buffer through which the bf16 planes are transposed, so that
// one warp instruction touches 8 rows x 64 contiguous bytes of global memory instead of 32 rows x 16 bytes
constexpr int kXposePitch = 80;
constexpr int kXposeWarpBytes = 32 * kXposePitch;
constexpr int kXposeBytes = 8 * kXposeWarpBytes;

struct GemmMaps {
  CUtensorMap a[3];
  CUtensorMap w[3];
  CUtensorMap out;   // TMA-store epilogue (single-plane bf16 output)
  CUtensorMap res;   // residual tile loads for that epilogue
};

struct GemmParams {
  int M, N;
  int taps, kw, cblocks;      // filter taps (kh*kw), filter width, 64-channel blocks per tap
  int n_terms;
  int term_a[kMaxGemmTerms], term_w[kMaxGemmTerms];
  int P, Q, stride, pad_h, pad_w;   // im2col geometry (output H, W)
  int num_m_tiles, num_n_tiles, stages;
  const float* scale;         // [N] or null (= 1)
  const float* bias;          // [N] or null (= 0)
  const __nv_bfloat16* res;   // residual planes [res_planes][M][ld_res] or null
  int ld_res, res_planes;
  long long res_plane_stride;
  __nv_bfloat16* out;         // [out_planes][M][ld_out] (+ out_col_off) or null
  int ld_out, out_col_off, out_planes;
  long long out_plane_stride;
  float* out_f32;             // [M][ld_out_f32] or null
  int ld_out_f32;
  int act;                    // 0 none, 1 relu, 2 gelu (erf)
  int tma_epi;                // 1: stage the bf16 output tile in shared memory and write it with TMA stores
  int n_out_bufs;             // 1 or 2 output staging tiles (2: the TMA store of tile i drains during tile i+1)
  int n_res_bufs;             // 0 or 2 residual staging tiles (the residual of tile i+1 is prefetched during tile i)
  int fast_gelu;              // 1: single-plane bf16 mode: act 2 is the tanh-form GELU (gelu_tanh_fast); 0: erf form
  int n_fastest;              // 1: consecutive tiles are the column blocks of one m-tile (round robin over the CTAs: the CTAs that
                              //    share an m-tile's A rows read them at the same time, one HBM read + L2 hits).  Default order is
                              //    m-fastest (a CTA keeps its column block, W tile and affine for many tiles): right while A fits L2
  int a_resident;             // 1: the A rows of an m-tile (all of K) stay in shared memory while the CTA walks that m-tile's
                              //    column blocks (tiles n-fastest, contiguous tile range per CTA); stages carry only W tiles
};

// exact-erf GELU of the tensor-core epilogues: erf by Abramowitz-Stegun 7.1.26 (|error| <= 2e-7 absolute: below the bf16
// rounding of a stored activation and at the level of the split-bf16 modes' own accumulation error) -- about half the instructions of erff(), whose two-branch evaluation made
// the fc1 + GELU layers of the ViTs ALU bound in their epilogue (129 us at 461 TFLOP/s for 50k x 1536 x 384).
DCR_DEVICE float gelu_erf_fast(float y) {
  const float ax = fabsf(y) * 0.70710678118654752440f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.f)));
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * ax * ax));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erf_abs = fmaf(-poly * t, e, 1.f);               // erf(|y| / sqrt 2)
  return 0.5f * y + 0.5f * fabsf(y) * erf_abs;                 // 0.5 y (1 + erf(y / sqrt 2)),  y erf(..) = |y| erf(|..|)
}

// GELU of the single-plane bf16 ("fast") mode: the tanh form with the hardware tanh -- 0.5 y (1 + tanh(0.79788 (y + 0.044715 y^3))),
// five FMA-pipe instructions and one MUFU per element.  It differs from the erf form by <= 4.7e-4 absolute (the form itself) plus
// <= 5e-4 |y| / 2 (tanh.approx.f32), below the bf16 rounding of the stored activation (2^-9 relative) for every |y| >= 0.1 and
// within two bf16 ulps below that.  The erf polynomial above costs 16 instructions and TWO MUFU ops per element: over a 128 x 256
// tile that is 4096 MUFU cycles against 3072 MMA cycles, which made fc1 + GELU epilogue bound (95 us at 627 TFLOP/s on ViT-S/16).
// The split-bf16 (fp32-level) modes and the float64 mode keep the erf forms.
DCR_DEVICE float gelu_tanh_fast(float y) {
  const float u = y * y;
  const float inner = y * fmaf(0.0356774081f, u, 0.7978845608f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(inner));
  const float h = 0.5f * y;
  return fmaf(h, t, h);
}

DCR_DEVICE float apply_act(float y, int act) {
  if (act == 1) return fmaxf(y, 0.f);
  if (act == 2) return gelu_erf_fast(y);                 // every tensor-core epilogue; the float64 mode (conv_exact.cu) keeps erff
  if (act == 3) return y / (1.f + expf(-1.702f * y));   // QuickGELU: x * sigmoid(1.702 x)  (CLIP, clip/model.py)
  return y;
}

DCR_DEVICE uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}

DCR_DEVICE void tmem_ld_wait_dep32(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                 "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                 "+r"(r[29]), "+r"(r[30]), "+r"(r[31])::"memory");
}

DCR_DEVICE void tma_store_2d(const void* tmap, const void* src_smem, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(smem_u32(src_smem)), "r"(c0), "r"(c1)
               : "memory");
}
DCR_DEVICE void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
DCR_DEVICE void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
DCR_DEVICE void tma_store_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
DCR_DEVICE void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// kEpi: 0 = direct epilogue (any number of planes, optional fp32 output, runtime activation; parity mode and final
//           layers), 1/2/3/4 = TMA-store epilogue with compile-time activation none / ReLU / GELU / QuickGELU (fast mode hot path).
// Eight epilogue warps: warps w and w+4 share a TMEM lane quadrant and split the tile's columns, so every SM
// sub-partition has two epilogue warps to switch between (the epilogue is latency bound, not issue bound).
//
// kCG == 2: two CTAs of a cluster (a TPC's SM pair) work one 256 x BN tile with UMMA 256 x BN x 16 (cta_group::2): each CTA
// loads its own 128 A rows and HALF of the W tile (BN/2 rows), the leader CTA issues the MMAs for both, each CTA's TMEM
// holds the accumulators of its own 128 rows and each runs its own epilogue.  Per CTA and k-block that is 16 KB + BN*64 B
// through the L2 -> shared-memory port instead of 16 KB + BN*128 B, and 4 KB + BN*16 B of operand reads per UMMA instead of
// 4 KB + BN*32 B -- the two resources the 128-wide single-CTA tiles are short of (DESIGN.md section 5d).  Plain (1x1 /
// Linear) single-term GEMMs with the TMA-store epilogue only; no A-resident mode.
template <int BN, bool kIm2col, int kEpi, int kCG>
__global__ void __launch_bounds__(kThreads, 1)
    gemm_bf16_kernel(const __grid_constant__ GemmMaps maps, const GemmParams p) {
  static_assert(kCG == 1 || (!kIm2col && kEpi != 0), "the CTA-pair form covers plain GEMMs with the TMA-store epilogue");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr bool kTma = kEpi != 0;
  constexpr int kBRows = BN / kCG;          // W rows this CTA loads per stage
  constexpr int kBStage = kBRows * kBK * 2;
  constexpr int kStageBytes = kAStage + kBStage;
  constexpr uint32_t kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  constexpr int kStagingBytes = (BN / 64) * kBM * 128;   // BN/64 slabs of [128 rows x 64 bf16], 128B swizzle
  constexpr int kChunksPerWarp = BN / 64;                // 32-column chunks each epilogue warp handles per tile
  const int stages = p.stages;
  const int k_iters = p.n_terms * p.taps * p.cblocks;
  // A-resident mode (wide 1x1 convolutions / Linear layers with small K): [k_iters x 16 KB A rows of the current m-tile]
  // first, then stages that carry only the W tile; the per-channel affine of ALL column blocks is staged once.
  const bool a_res = (kCG == 1) && p.a_resident != 0;
  const int stage_bytes = a_res ? kBStage : kStageBytes;
  const int num_n_tiles = p.num_n_tiles;
  uint8_t* smem_ares = smem;
  uint8_t* smem_ab = smem + (a_res ? k_iters * kAStage : 0);
  uint8_t* out_stage = smem_ab + stages * stage_bytes;                      // n_out_bufs tiles, 1024-aligned
  // direct epilogue (kEpi == 0): no staging tiles; one 32-row x 64-byte transpose buffer per epilogue warp instead
  uint8_t* res_stage = out_stage + (kTma ? p.n_out_bufs * kStagingBytes : kXposeBytes);   // n_res_bufs tiles
  float* sb = reinterpret_cast<float*>(res_stage + p.n_res_bufs * kStagingBytes);   // [2 bufs][2 (scale,bias)][BN] | a_res: [2][n_tiles*BN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sb + (a_res ? 2 * num_n_tiles * BN : 4 * BN));
  uint64_t* full = bars;          // [stages] (<= 12)
  uint64_t* empty = bars + 12;    // [stages]
  uint64_t* t_full = bars + 24;   // [2]
  uint64_t* t_empty = bars + 26;  // [2]
  uint64_t* res_full = bars + 28;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 30);
  uint64_t* a_full = bars + 10;    // A-resident mode (stages <= 8, so full[10..11] are free)
  uint64_t* a_empty = bars + 11;

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // hoist everything the tile loops need out of the constant bank once
  const int M = p.M, N = p.N, num_m_tiles = p.num_m_tiles;
  const bool has_res = p.res != nullptr;
  // CTA pair: tiles are 2 m-tiles tall, the pair (cluster) is the scheduling unit and CTA rank r works m-tile 2*pm + r (an
  // odd last m-tile leaves rank 1 a tile past M: its loads are zero filled, its stores skipped)
  const uint32_t cta_rank = (kCG == 2) ? cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int pair_m_tiles = (num_m_tiles + kCG - 1) / kCG;
  const int num_tiles = pair_m_tiles * p.num_n_tiles;
  const int unit = static_cast<int>(blockIdx.x) / kCG, n_units = static_cast<int>(gridDim.x) / kCG;
  // tile sequence of this CTA: m-fastest round robin (default) or a contiguous range of the n-fastest order (A-resident)
  const int t_first = a_res ? static_cast<int>(static_cast<long long>(num_tiles) * blockIdx.x / gridDim.x) : unit;
  const int t_end = a_res ? static_cast<int>(static_cast<long long>(num_tiles) * (blockIdx.x + 1) / gridDim.x) : num_tiles;
  const int t_step = a_res ? 1 : n_units;
  const bool n_fast = p.n_fastest != 0;
  auto tile_m = [&](int t) {
    return a_res ? t / num_n_tiles : ((n_fast ? t / num_n_tiles : t % pair_m_tiles) * kCG + static_cast<int>(cta_rank));
  };
  auto tile_n = [&](int t) { return (a_res || n_fast) ? t % num_n_tiles : t / pair_m_tiles; };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.out);
    tma_prefetch_desc(&maps.res);
    for (int i = 0; i < 3; ++i) {
      tma_prefetch_desc(&maps.a[i]);
      tma_prefetch_desc(&maps.w[i]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full[s], kCG);        // pair: the leader's barrier takes one arrive per CTA and both CTAs' bytes
      mbar_init(&empty[s], 1);         // pair: tcgen05.commit multicasts the arrive to both CTAs
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&t_full[b], 1);
      mbar_init(&t_empty[b], 8 * kCG);   // pair: the leader's MMA warp waits for both CTAs' epilogue warps
      mbar_init(&res_full[b], 1);
    }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc<kCG>(tmem_slot, kTmemCols);
    tmem_relinquish<kCG>();
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (kCG == 2) cluster_sync();   // the peer's barriers are initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Producer and MMA roles: the WHOLE warp walks the loops (so that every value is provably warp-uniform and lives
  // in uniform registers) and one elected lane issues the TMA / tcgen05 instructions.  Running the loops under
  // `if (lane == 0)` makes the compiler wrap every UTMALDG / UTCHMMA in an ELECT + R2UR.BROADCAST + BRA.U.ANY loop
  // (8-20 extra instructions each) -- and the single-thread instruction stream IS the pipeline's critical path.
  if (warp == 0) {
    {
      const int n_terms = p.n_terms, taps = p.taps, kw = p.kw, cblocks = p.cblocks;
      PipeState st(stages);
      int res_m = -1;
      uint32_t a_seg = 0;
      for (int tile = t_first; tile < t_end; tile += t_step) {
        const int m0 = tile_m(tile) * kBM;
        const int n0 = tile_n(tile) * BN;
        if (a_res) {
          if (m0 != res_m) {   // new m-tile: its A rows (all of K) once, after the MMAs on the previous rows have retired
            res_m = m0;
            mbar_wait(a_empty, (a_seg & 1) ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(a_full, k_iters * kAStage);
              for (int ki = 0; ki < k_iters; ++ki)
                tma_load_2d<1>(smem_ares + ki * kAStage, &maps.a[p.term_a[0]], a_full, ki * kBK, m0, kEvictFirst);
            }
            __syncwarp();
            ++a_seg;
          }
          for (int ki = 0; ki < k_iters; ++ki, st.next()) {
            const uint32_t s = st.s;
            mbar_wait(&empty[s], st.ph ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&full[s], kBStage);
              tma_load_2d<1>(smem_ab + s * kBStage, &maps.w[p.term_w[0]], &full[s], ki * kBK, n0, kEvictLast);
            }
            __syncwarp();
          }
          continue;
        }
        int img = 0, h0 = 0, w0 = 0;
        if constexpr (kIm2col) {
          const int pq = p.P * p.Q;
          img = m0 / pq;
          const int rem = m0 - img * pq;
          const int p0 = rem / p.Q, q0 = rem - p0 * p.Q;
          h0 = p0 * p.stride - p.pad_h;
          w0 = q0 * p.stride - p.pad_w;
        }
        for (int t = 0; t < n_terms; ++t) {
          const CUtensorMap* ma = &maps.a[p.term_a[t]];
          const CUtensorMap* mw = &maps.w[p.term_w[t]];
          for (int tap = 0; tap < taps; ++tap) {
            const int r = tap / kw, sx = tap - r * kw;
            for (int cb = 0; cb < cblocks; ++cb, st.next()) {
              const uint32_t s = st.s, ph = st.ph;
              mbar_wait(&empty[s], ph ^ 1);
              if (elect_one()) {
                if (leader) mbar_arrive_expect_tx(&full[s], kStageBytes * kCG);
                else mbar_arrive_cluster(&full[s], 0);
                uint8_t* sa = smem_ab + s * kStageBytes;
                if constexpr (kIm2col)
                  tma_load_im2col_4d<1>(sa, ma, &full[s], cb * kBK, w0, h0, img, static_cast<uint16_t>(sx),
                                        static_cast<uint16_t>(r));
                else
                  tma_load_2d<kCG>(sa, ma, &full[s], cb * kBK, m0, kEvictNormal);
                tma_load_2d<kCG>(sa + kAStage, mw, &full[s], (tap * cblocks + cb) * kBK, n0 + static_cast<int>(cta_rank) * kBRows,
                                 kEvictNormal);
              }
              __syncwarp();
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(kBM * kCG, BN);
      uint32_t tc = 0;
      PipeState st(stages);
      // descriptors of stage 0; stage s adds s * kStageBytes to the 16-byte-granular start-address field (no carry out
      // of the field: shared memory addresses stay below 256 KB)
      const uint64_t da0 = umma_desc_sw128(smem_u32(a_res ? smem_ares : smem_ab));
      const uint64_t db0 = umma_desc_sw128(smem_u32(a_res ? smem_ab : smem_ab + kAStage));
      const uint32_t a_step = a_res ? (kAStage >> 4) : (kStageBytes >> 4);     // A: per k-iteration (resident) / per stage
      const uint32_t b_step = static_cast<uint32_t>(stage_bytes) >> 4;
      int res_m = -1;
      uint32_t a_seg = 0;
      for (int tile = t_first; tile < t_end; tile += t_step, ++tc) {
        const uint32_t buf = tc & 1;
        bool last_of_m = false;
        if (a_res) {
          const int m = tile_m(tile);
          if (m != res_m) {
            res_m = m;
            mbar_wait(a_full, a_seg & 1);
            tc_fence_after();
            ++a_seg;
          }
          last_of_m = (tile + 1 >= t_end) || tile_m(tile + 1) != m;
        }
        mbar_wait(&t_empty[buf], ((tc >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * BN;
        for (int ki = 0; ki < k_iters; ++ki, st.next()) {
          const uint32_t s = st.s;
          mbar_wait(&full[s], st.ph);
          tc_fence_after();
          const uint64_t da = da0 + static_cast<uint64_t>((a_res ? static_cast<uint32_t>(ki) : s) * a_step);
          const uint64_t db = db0 + static_cast<uint64_t>(s * b_step);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k) umma_f16<kCG>(tmem_d, da + 2 * k, db + 2 * k, idesc, (ki | k) != 0);
            umma_commit<kCG>(&empty[s]);
            if (ki == k_iters - 1) {
              umma_commit<kCG>(&t_full[buf]);
              if (last_of_m) umma_commit<kCG>(a_empty);
            }
          }
          __syncwarp();
        }
      }
    }
  } else {
    const uint32_t ewarp = warp - 2;               // 0..7
    const uint32_t quad = warp & 3;                // TMEM lane quadrant
    const uint32_t half = ewarp >> 2;              // which half of the tile's columns
    const uint32_t row = quad * 32 + lane;
    const uint32_t etid = ewarp * 32 + lane;       // 0..255 among the epilogue threads
    const uint32_t tmem_row = tmem_base + ((quad * 32u) << 16);
    const int act = p.act;
    uint32_t tc = 0;
    auto load_residual = [&](int tile_idx, uint32_t rbuf) {   // one thread: residual tile -> res_stage[rbuf]
      const int rm0 = tile_m(tile_idx) * kBM;
      const int rn0 = tile_n(tile_idx) * BN;
      int slabs = 0;
      for (int sl = 0; sl < BN / 64; ++sl)
        if (rn0 + sl * 64 < N) ++slabs;
      mbar_arrive_expect_tx(&res_full[rbuf], slabs * kBM * 128);
      for (int sl = 0; sl < BN / 64; ++sl)
        if (rn0 + sl * 64 < N)
          tma_load_2d<1>(res_stage + rbuf * kStagingBytes + sl * kBM * 128, &maps.res, &res_full[rbuf], rn0 + sl * 64, rm0,
                         kEvictFirst);
    };
    if (kTma && has_res && etid == 0 && t_first < t_end) load_residual(t_first, 0);
    const bool two_out = p.n_out_bufs == 2;
    const uint32_t sb_addr = smem_u32(sb), out_addr = smem_u32(out_stage), res_addr = smem_u32(res_stage);
    int staged_n0 = -1;
    uint32_t sbsel = 1;
    if (a_res) {   // per-channel affine of every column block, once
      const int npad = num_n_tiles * BN;
      for (int c = etid; c < npad; c += 256) {
        st_shared_f32(sb_addr + c * 4, (p.scale && c < N) ? p.scale[c] : 1.f);
        st_shared_f32(sb_addr + (npad + c) * 4, (p.bias && c < N) ? p.bias[c] : 0.f);
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    for (int tile = t_first; tile < t_end; tile += t_step, ++tc) {
      const int m0 = tile_m(tile) * kBM;
      const int n0 = tile_n(tile) * BN;
      const uint32_t buf = tc & 1;
      uint8_t* ostage = out_stage + (two_out ? (tc & 1) : 0) * kStagingBytes;
      const uint32_t ostage_addr = out_addr + (two_out ? (tc & 1) : 0) * kStagingBytes;
      const uint32_t rstage_addr = res_addr + (tc & 1) * kStagingBytes;
      if constexpr (kTma) {
        if (etid == 0) {
          // single output staging tile: it is free once the store of the previous tile has finished READING it (with
          // two tiles that wait sits before the end-of-tile barrier, see below)
          if (!two_out) tma_store_wait_read();
          // prefetch the NEXT tile's residual; its buffer was last read in tile tc-1 (all warps passed that barrier)
          if (has_res && tile + t_step < t_end) load_residual(tile + t_step, (tc & 1) ^ 1);
        }
      }
      // Per-channel affine: staged only when the column block changes (tiles are walked m-fastest, so a CTA keeps its
      // column block for many tiles) into the buffer the previous block did not use -- warps still finishing the
      // previous tile read the other one.  The barrier is also what orders a single output staging tile's reuse.
      const bool restage = !a_res && n0 != staged_n0;
      if (restage) {
        sbsel ^= 1;
        staged_n0 = n0;
        for (int c = etid; c < BN; c += 256) {
          const int n = n0 + c;
          st_shared_f32(sb_addr + (sbsel * 2 * BN + c) * 4, (p.scale && n < N) ? p.scale[n] : 1.f);
          st_shared_f32(sb_addr + (sbsel * 2 * BN + BN + c) * 4, (p.bias && n < N) ? p.bias[n] : 0.f);
        }
      }
      if (restage || (kTma && !two_out)) asm volatile("bar.sync 1, 256;" ::: "memory");
      const uint32_t s_scale = a_res ? sb_addr + n0 * 4 : sb_addr + sbsel * 2 * BN * 4;
      const uint32_t s_bias = s_scale + (a_res ? num_n_tiles * BN : BN) * 4;
      mbar_wait(&t_full[buf], (tc >> 1) & 1);
      tc_fence_after();
      if (kTma && has_res) mbar_wait(&res_full[tc & 1], (tc >> 1) & 1);
      const int m = m0 + static_cast<int>(row);
      const bool row_ok = m < M;
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
          if (lane == 0) {
            if constexpr (kCG == 2) mbar_arrive_cluster(&t_empty[buf], 0);
            else mbar_arrive(&t_empty[buf]);
          }
        }
        const int nc = n0 + ch * 32;
        if (nc >= N) continue;
        float y[32];
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const float4 sc = ld_shared_f4(s_scale + (ch * 32 + c) * 4);
          const float4 bi = ld_shared_f4(s_bias + (ch * 32 + c) * 4);
          y[c + 0] = fmaf(__uint_as_float(r[c + 0]), sc.x, bi.x);
          y[c + 1] = fmaf(__uint_as_float(r[c + 1]), sc.y, bi.y);
          y[c + 2] = fmaf(__uint_as_float(r[c + 2]), sc.z, bi.z);
          y[c + 3] = fmaf(__uint_as_float(r[c + 3]), sc.w, bi.w);
        }
        if constexpr (kTma) {
          // this thread's 32 columns live in slab ch/2 at 16-byte chunks (ch&1)*4 .. +3 of row `row` (128B swizzle)
          const uint32_t srow = ostage_addr + (ch >> 1) * kBM * 128 + row * 128;
          const uint32_t rrow = rstage_addr + (ch >> 1) * kBM * 128 + row * 128;
          const uint32_t sw = row & 7;
          if (has_res) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 rv = ld_shared_v4(rrow + ((((ch & 1) * 4 + j) ^ sw) << 4));
              const uint32_t w[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                y[j * 8 + 2 * e] += __uint_as_float(w[e] << 16);
                y[j * 8 + 2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u);
              }
            }
          }
#pragma unroll
          for (int c = 0; c < 32; ++c) y[c] = (kEpi == 3) ? gelu_tanh_fast(y[c]) : apply_act(y[c], kEpi - 1);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 v;
            v.x = pack_bf16(y[j * 8 + 0], y[j * 8 + 1]);
            v.y = pack_bf16(y[j * 8 + 2], y[j * 8 + 3]);
            v.z = pack_bf16(y[j * 8 + 4], y[j * 8 + 5]);
            v.w = pack_bf16(y[j * 8 + 6], y[j * 8 + 7]);
            st_shared_v4(srow + ((((ch & 1) * 4 + j) ^ sw) << 4), v);
          }
        } else {
          // Direct epilogue (split-bf16 planes, fp32 outputs, final layers).  Thread = accumulator row, but a row's 32 columns
          // are only 64 bytes per plane: written straight from the registers, one warp instruction touched 32 rows x 16 bytes
          // (32 half-used sectors, 32 LSU wavefronts) and the 1x1 expansions of the fp32-level modes ran at 0.5 TB/s (layer1:
          // 870 us against 97 us with the TMA-store epilogue in one-plane mode).  Every plane now goes through the warp's
          // transpose buffer: rows -> shared memory, then 8 rows x 64 contiguous bytes per instruction to / from global memory.
          const int nvalid = min(32, N - nc);   // multiple of 8 (N % 8 == 0 enforced on the host)
          const uint32_t xw = smem_u32(out_stage) + ewarp * kXposeWarpBytes;
          const uint32_t x_own = xw + lane * kXposePitch;           // this thread's row
          const int m_w0 = m0 + static_cast<int>(quad) * 32;        // first row of this warp
          if (has_res) {
            for (int pl = 0; pl < p.res_planes; ++pl) {
              const __nv_bfloat16* rbase = p.res + pl * p.res_plane_stride + nc;
              __syncwarp();
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const int piece = t * 32 + static_cast<int>(lane), r = piece >> 2, part = piece & 3;
                if (m_w0 + r < M && part * 8 < nvalid)
                  st_shared_v4(xw + r * kXposePitch + part * 16,
                               *reinterpret_cast<const uint4*>(rbase + static_cast<size_t>(m_w0 + r) * p.ld_res + part * 8));
              }
              __syncwarp();
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (j * 8 < nvalid && row_ok) {
                  const uint4 rv = ld_shared_v4(x_own + j * 16);
                  const uint32_t w[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    y[j * 8 + 2 * e] += __uint_as_float(w[e] << 16);
                    y[j * 8 + 2 * e + 1] += __uint_as_float(w[e] & 0xffff0000u);
                  }
                }
              }
            }
          }
          // the activation is a run-time value here: ONE warp-uniform switch per chunk (inside the element loop the compiler
          // kept a compare-and-branch chain per element: 660 instructions per 32-column chunk, a quarter of the warp samples on
          // instruction fetch)
          if (act == 1) {
#pragma unroll
            for (int c = 0; c < 32; ++c) y[c] = fmaxf(y[c], 0.f);
          } else if (act == 2) {
            if (p.fast_gelu) {
#pragma unroll
              for (int c = 0; c < 32; ++c) y[c] = gelu_tanh_fast(y[c]);
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c) y[c] = gelu_erf_fast(y[c]);
            }
          } else if (act == 3) {
#pragma unroll
            for (int c = 0; c < 32; ++c) y[c] = apply_act(y[c], 3);
          }
          if (p.out_f32 && row_ok) {
            float* op = p.out_f32 + static_cast<size_t>(m) * p.ld_out_f32 + nc;
#pragma unroll
            for (int c = 0; c < 32; c += 4)
              if (c < nvalid) *reinterpret_cast<float4*>(op + c) = make_float4(y[c], y[c + 1], y[c + 2], y[c + 3]);
          }
          if (p.out) {
            for (int pl = 0; pl < p.out_planes; ++pl) {
              __nv_bfloat16* obase = p.out + pl * p.out_plane_stride + p.out_col_off + nc;
              __syncwarp();
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                uint4 v;
                v.x = pack_bf16(y[j * 8 + 0], y[j * 8 + 1]);
                v.y = pack_bf16(y[j * 8 + 2], y[j * 8 + 3]);
                v.z = pack_bf16(y[j * 8 + 4], y[j * 8 + 5]);
                v.w = pack_bf16(y[j * 8 + 6], y[j * 8 + 7]);
                st_shared_v4(x_own + j * 16, v);
              }
              __syncwarp();
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const int piece = t * 32 + static_cast<int>(lane), r = piece >> 2, part = piece & 3;
                if (m_w0 + r < M && part * 8 < nvalid)
                  *reinterpret_cast<uint4*>(obase + static_cast<size_t>(m_w0 + r) * p.ld_out + part * 8) =
                      ld_shared_v4(xw + r * kXposePitch + part * 16);
              }
              if (pl + 1 < p.out_planes) {
                // next plane holds the rounding residual of this one
#pragma unroll
                for (int c = 0; c < 32; ++c) y[c] -= __bfloat162float(__float2bfloat16_rn(y[c]));
              }
            }
          }
        }
      }
      if constexpr (kTma) {
        fence_proxy_async();   // generic-proxy writes -> visible to the TMA (async proxy)
        // two output staging tiles: the NEXT tile writes the tile the PREVIOUS store (committed a whole tile ago) reads
        // from; that read must be over before anyone passes this barrier
        if (two_out && etid == 0) tma_store_wait_read();
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (etid == 0) {
          for (int sl = 0; sl < BN / 64; ++sl)
            if (n0 + sl * 64 < N && m0 < M) tma_store_2d(&maps.out, ostage + sl * kBM * 128, p.out_col_off + n0 + sl * 64, m0);
          tma_store_commit();
        }
      }
    }
  }

  if (kTma && warp == 2 && lane == 0) tma_store_wait_all();   // etid 0 issued the stores
  tc_fence_before();
  __syncthreads();
  if constexpr (kCG == 2) cluster_sync();   // the peer's MMAs (issued by the leader) read this CTA's tiles and write its TMEM
  if (warp == 2) tmem_dealloc<kCG>(tmem_base, kTmemCols);
}

// A-resident mode: plain (non-im2col) single-term GEMMs with several column blocks and K <= 256 -- the wide 1x1
// expansions: the A rows of an m-tile are loaded once instead of once per column block (per-SM-unique data is what
// the L2 -> shared-memory path is short of; the W tiles are shared by all SMs and cheap)
// (the resident rows are single buffered: the next m-tile's rows wait for the last MMA on the current ones, a bubble
// that only pays off when the epilogue is heavy (residual) or the m-tile has >= 4 column blocks; measured on B200,
// batch 256: 177 -> 157 us for the layer1 expansion with residual, 98 -> 90 us layer2, but 103 -> 130 us for the
// residual-free 2-block downsample)
bool wants_a_resident(const GemmParams& p, int BN, bool im2col, size_t max_smem) {
  const int k_iters_h = p.n_terms * p.taps * p.cblocks;
  if (!(!im2col && p.tma_epi && p.n_terms == 1 && p.num_n_tiles >= 2 && (p.res != nullptr || p.num_n_tiles >= 4) &&
        k_iters_h * kAStage <= 64 * 1024 && p.num_n_tiles * BN <= 4096))
    return false;
  // the resident rows, the all-blocks affine table and the staging tiles must leave at least three W stages; otherwise
  // the layer runs with the default schedule
  const size_t staging = static_cast<size_t>(BN / 64) * kBM * 128;
  const size_t need = 1024 + static_cast<size_t>(2) * p.num_n_tiles * BN * 4 + static_cast<size_t>(k_iters_h) * kAStage + 256 +
                      static_cast<size_t>(1 + (p.res ? 2 : 0)) * staging + 3 * static_cast<size_t>(BN) * kBK * 2;
  return need <= max_smem;
}

template <int BN, bool kIm2col, int kEpi, int kCG>
int launch(const GemmMaps& maps, GemmParams& p, int num_sms, size_t max_smem, cudaStream_t stream) {
  constexpr int kStageBytes = kAStage + (BN / kCG) * kBK * 2;
  constexpr size_t kStagingBytes = static_cast<size_t>(BN / 64) * kBM * 128;
  // staging tiles: residual layers get 2 residual + 2 output tiles (prefetch / drain a full tile ahead) when they still
  // leave >= 3 pipeline stages, otherwise one output tile (plus two residual tiles if needed)
  p.n_res_bufs = (p.tma_epi && p.res) ? 2 : 0;
  p.n_out_bufs = p.tma_epi ? 2 : 0;
  const int k_iters_h = p.n_terms * p.taps * p.cblocks;
  p.a_resident = (kCG == 1 && kEpi != 0 && wants_a_resident(p, BN, kIm2col, max_smem)) ? 1 : 0;
  const size_t sb_bytes = p.a_resident ? static_cast<size_t>(2) * p.num_n_tiles * BN * 4 : static_cast<size_t>(4) * BN * 4;
  const size_t ares_bytes = p.a_resident ? static_cast<size_t>(k_iters_h) * kAStage : 0;
  auto fixed_for = [&](int nout, int nres) {
    return 1024 + sb_bytes + ares_bytes + 256 + static_cast<size_t>(nout + nres) * kStagingBytes + (p.tma_epi ? 0 : kXposeBytes);
  };
  const size_t stage_bytes = p.a_resident ? static_cast<size_t>(BN) * kBK * 2 : static_cast<size_t>(kStageBytes);
  if (p.tma_epi && (fixed_for(p.n_out_bufs, p.n_res_bufs) + 3 * stage_bytes > max_smem)) p.n_out_bufs = 1;
  const size_t fixed = fixed_for(p.n_out_bufs, p.n_res_bufs);
  DCR_REQUIRE(max_smem > fixed + 2 * stage_bytes, "gemm: not enough shared memory");
  int stages = static_cast<int>((max_smem - fixed) / stage_bytes);
  stages = std::min(stages, 8);
  p.stages = stages;
  const size_t smem = fixed + static_cast<size_t>(stages) * stage_bytes;
  auto kern = gemm_bf16_kernel<BN, kIm2col, kEpi, kCG>;
  static bool attr_set_dev[64] = {};   // per template instantiation and device (the attribute is per device)
  int cur_dev = 0;
  DCR_CUDA_CHECK(cudaGetDevice(&cur_dev));
  bool& attr_set = attr_set_dev[cur_dev & 63];
  if (!attr_set) {
    DCR_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(max_smem)));
    attr_set = true;
  }
  if constexpr (kCG == 2) {
    const int pair_tiles = ((p.num_m_tiles + 1) / 2) * p.num_n_tiles;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * std::min(pair_tiles, num_sms / 2));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    DCR_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, maps, p));
  } else {
    const int tiles = p.num_m_tiles * p.num_n_tiles;
    const int grid = std::min(tiles, num_sms);
    kern<<<grid, kThreads, smem, stream>>>(maps, p);
  }
  count_launch();
  DCR_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

int conv_gemm(const ConvGemmDesc& d, cudaStream_t stream) {
  const DeviceInfo* di = device_info();
  if (!di) return -2;
  DCR_REQUIRE(di->cc_major == 10, "conv_gemm: this build targets sm_100a; device reports sm_%d%d", di->cc_major, di->cc_minor);
  DCR_REQUIRE(d.n_terms >= 1 && d.n_terms <= kMaxGemmTerms, "conv_gemm: bad n_terms %d", d.n_terms);
  DCR_REQUIRE(d.C % 8 == 0 && d.N % 8 == 0, "conv_gemm: C (%d) and N (%d) must be multiples of 8", d.C, d.N);
  DCR_REQUIRE(d.kh >= 1 && d.kw >= 1 && d.stride >= 1, "conv_gemm: bad filter geometry");
  DCR_REQUIRE(d.act >= 0 && d.act <= 3, "conv_gemm: unknown activation %d", d.act);
  if (d.exact) return conv_exact(d, stream);
  if (conv3x3_halo_eligible(d)) return conv3x3_halo(d, stream);
  const bool windowed = d.in_stride_w != 0;
  const bool im2col = windowed || !(d.kh == 1 && d.kw == 1 && d.stride == 1 && d.pad_h == 0 && d.pad_w == 0);
  const int P = (d.H + 2 * d.pad_h - d.kh) / d.stride + 1;
  const int Q = (d.W + 2 * d.pad_w - d.kw) / d.stride + 1;
  const long long M = static_cast<long long>(d.B) * P * Q;
  DCR_REQUIRE(M > 0 && M < (1ll << 31), "conv_gemm: M out of range");
  const int cblocks = (d.C + kBK - 1) / kBK;
  const int ktot = d.kh * d.kw * cblocks * kBK;   // padded K of the prepared weights

  GemmMaps maps;
  memset(&maps, 0, sizeof(maps));
  int a_planes = 0, w_planes = 0;
  for (int t = 0; t < d.n_terms; ++t) {
    a_planes = std::max(a_planes, d.term_a[t] + 1);
    w_planes = std::max(w_planes, d.term_w[t] + 1);
  }
  DCR_REQUIRE(a_planes <= 3 && w_planes <= 3, "conv_gemm: at most 3 planes");
  int BN = d.N <= 64 ? 64 : (d.N <= 128 ? 128 : 256);
  // memory-bound shapes (residual epilogue, or little K per output) favour 128-wide tiles: their staging tiles can be
  // double buffered; compute-bound shapes keep 256 (fewer re-reads of A)
  const bool single_plane = d.out && d.out_planes <= 1 && !d.out_f32 && (!d.res || d.res_planes <= 1);
  if (BN == 256 && single_plane && (d.res != nullptr || static_cast<long long>(d.kh) * d.kw * d.C <= 256)) BN = 128;
  // (256-wide tiles for the long-K residual layers -- ResNet layer4 expansions, K = 512 -- were tried in round 2: the output
  // and residual staging tiles of a 128 x 256 tile do not fit beside three pipeline stages)
  // few output tiles and a long K (the SSCD head: 256 x 512 x 2048 is four 128 x 256 tiles, each CTA streaming 1.5 MB through
  // one SM's L2 port: 22 us): narrower tiles put more CTAs -- more L2 ports -- on the same K stream
  {
    const long long m_tiles = (M + kBM - 1) / kBM;
    while (BN > 64 && ktot >= 1024 && m_tiles * ((d.N + BN - 1) / BN) * 4 <= di->num_sms) BN /= 2;
  }
  for (int pl = 0; pl < 3; ++pl) {
    const int pa = std::min(pl, a_planes - 1), pw = std::min(pl, w_planes - 1);
    const __nv_bfloat16* abase = d.in + pa * d.in_plane_stride;
    if (im2col) {
      DCR_REQUIRE(windowed || d.ld_in == d.C, "conv_gemm: im2col input must be dense NHWC (ld_in == C)");
      if (int rc = make_tmap_im2col_bf16(&maps.a[pl], abase, d.B, d.H, d.W, d.C, d.pad_h, d.pad_w, d.kh, d.kw, d.stride,
                                         kBK, kBM, d.in_stride_w, d.in_stride_h, d.in_stride_n))
        return rc;
    } else {
      if (int rc = make_tmap_2d_bf16(&maps.a[pl], abase, M, d.C, d.ld_in, kBM, kBK)) return rc;
    }
    if (int rc = make_tmap_2d_bf16(&maps.w[pl], d.weight + pw * d.w_plane_stride, d.N, ktot, ktot, BN, kBK)) return rc;
  }

  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = static_cast<int>(M);
  p.N = d.N;
  p.taps = d.kh * d.kw;
  p.kw = d.kw;
  p.cblocks = cblocks;
  p.n_terms = d.n_terms;
  for (int t = 0; t < d.n_terms; ++t) {
    p.term_a[t] = d.term_a[t];
    p.term_w[t] = d.term_w[t];
  }
  p.P = P;
  p.Q = Q;
  p.stride = d.stride;
  p.pad_h = d.pad_h;
  p.pad_w = d.pad_w;
  p.num_m_tiles = static_cast<int>((M + kBM - 1) / kBM);
  p.num_n_tiles = (d.N + BN - 1) / BN;
  p.scale = d.scale;
  p.bias = d.bias;
  p.res = d.res;
  p.ld_res = d.ld_res;
  p.res_planes = d.res ? std::max(1, d.res_planes) : 0;
  p.res_plane_stride = d.res_plane_stride;
  p.out = d.out;
  p.ld_out = d.ld_out;
  p.out_col_off = d.out_col_off;
  p.out_planes = d.out ? std::max(1, d.out_planes) : 0;
  p.out_plane_stride = d.out_plane_stride;
  p.out_f32 = d.out_f32;
  p.ld_out_f32 = d.ld_out_f32;
  p.act = d.act;
  p.fast_gelu = (d.n_terms == 1 && p.out_planes <= 1) ? 1 : 0;
  // tile order: with several column blocks and an A matrix larger than what L2 keeps between the passes, m-fastest order
  // streams A from HBM once per column block (ViT-S fc2: 155 MB x 3 = 83 us of HBM time for a 99 us layer)
  const double a_bytes = 2.0 * a_planes * (im2col ? static_cast<double>(d.B) * d.H * d.W * d.C : static_cast<double>(M) * d.C);
  const int order = tuning_int("DCR_GEMM_TILE_ORDER", -1);   // tuning / tests: 0 = m-fastest, 1 = n-fastest, default by size
  p.n_fastest = (order >= 0) ? (order == 1 && p.num_n_tiles >= 2) : (p.num_n_tiles >= 2 && a_bytes > 48e6);
  p.tma_epi = (p.out != nullptr && p.out_planes == 1 && p.out_f32 == nullptr && (p.res == nullptr || p.res_planes == 1) &&
               (d.act != 2 || p.fast_gelu))   // the TMA-store epilogue's compile-time GELU is the tanh form
                  ? 1
                  : 0;
  if (p.tma_epi) {
    // dim0 = col_off + N so that a partial last slab is clipped at this op's own columns (concat neighbours intact)
    if (int rc = make_tmap_2d_bf16(&maps.out, p.out, M, p.out_col_off + d.N, p.ld_out, kBM, 64)) return rc;
    if (p.res) {
      if (int rc = make_tmap_2d_bf16(&maps.res, p.res, M, d.N, p.ld_res, kBM, 64)) return rc;
    } else {
      maps.res = maps.out;
    }
  } else {
    maps.out = maps.w[0];
    maps.res = maps.w[0];
  }
  DCR_REQUIRE(p.out == nullptr || (p.ld_out % 8 == 0 && p.out_col_off % 8 == 0), "conv_gemm: output leading dim / offset must be multiples of 8");
  DCR_REQUIRE(p.res == nullptr || p.ld_res % 8 == 0, "conv_gemm: residual leading dim must be a multiple of 8");
  DCR_REQUIRE(p.out_f32 == nullptr || p.ld_out_f32 % 4 == 0, "conv_gemm: fp32 output leading dim must be a multiple of 4");

  // ---- CTA-pair form (cta_group::2, 256-row tiles, half a W tile per CTA): plain single-term GEMMs with the TMA-store
  // epilogue whose A rows are not kept resident and that have enough m-tiles to fill the pairs
  const int want_cg2 = tuning_int("DCR_GEMM_CG2", -1);   // 0: never, 1: wherever the kernel form exists, default: policy
  bool use_cg2 = !im2col && p.tma_epi && p.n_terms == 1 && (BN == 128 || BN == 256) && want_cg2 != 0;
  if (use_cg2 && want_cg2 < 0) {
    // measured per layer at batch 256 (tools/pair_bench.py, B200): 256-wide tiles gain 5-11 % from K = 384 up (ResNet layer3/4
    // reductions 256<-1024, 512<-1024; ViT qkv 1152<-384, ViT-B qkv / fc1); 128-wide residual tiles gain only with many column
    // blocks and K >= 512 (layer4 expansion 2048<-512: 9 %; ViT fc2 / proj with 3 column blocks: none); short K loses
    const long long pair_tiles = static_cast<long long>((p.num_m_tiles + 1) / 2) * p.num_n_tiles;
    const bool shape_ok = (BN == 256) ? ktot >= 384 : (ktot >= 512 && p.num_n_tiles >= 8);
    use_cg2 = !wants_a_resident(p, BN, im2col, di->max_smem_optin) && shape_ok && pair_tiles >= di->num_sms;
  }
  if (use_cg2) {
    for (int pl = 0; pl < 3; ++pl) {
      const int pw = std::min(pl, w_planes - 1);
      if (int rc = make_tmap_2d_bf16(&maps.w[pl], d.weight + pw * d.w_plane_stride, d.N, ktot, ktot, BN / 2, kBK)) return rc;
    }
  }
  const int epi = p.tma_epi ? 1 + p.act : 0;   // compile-time activation on the TMA-store path
  if (use_cg2) {
#define DCR_LAUNCH_PAIR(BNv)                                                                                     \
  (epi == 1 ? launch<BNv, false, 1, 2>(maps, p, di->num_sms, di->max_smem_optin, stream)                         \
            : (epi == 2 ? launch<BNv, false, 2, 2>(maps, p, di->num_sms, di->max_smem_optin, stream)             \
                        : (epi == 3 ? launch<BNv, false, 3, 2>(maps, p, di->num_sms, di->max_smem_optin, stream) \
                                    : launch<BNv, false, 4, 2>(maps, p, di->num_sms, di->max_smem_optin, stream))))
    return BN == 128 ? DCR_LAUNCH_PAIR(128) : DCR_LAUNCH_PAIR(256);
#undef DCR_LAUNCH_PAIR
  }

#define DCR_LAUNCH_E(BNv, E)                                                                      \
  (im2col ? launch<BNv, true, E, 1>(maps, p, di->num_sms, di->max_smem_optin, stream)              \
          : launch<BNv, false, E, 1>(maps, p, di->num_sms, di->max_smem_optin, stream))
#define DCR_LAUNCH(BNv)                                                                          \
  (epi == 0 ? DCR_LAUNCH_E(BNv, 0)                                                                \
            : (epi == 1 ? DCR_LAUNCH_E(BNv, 1) : (epi == 2 ? DCR_LAUNCH_E(BNv, 2) : (epi == 3 ? DCR_LAUNCH_E(BNv, 3) : DCR_LAUNCH_E(BNv, 4)))))
  switch (BN) {
    case 64: return DCR_LAUNCH(64);
    case 128: return DCR_LAUNCH(128);
    case 256: return DCR_LAUNCH(256);
    default: return set_error(-1, "conv_gemm: unsupported BN %d", BN);
  }
#undef DCR_LAUNCH_E
#undef DCR_LAUNCH
}

}  // namespace dcr
