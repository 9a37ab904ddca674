// Internal C++ declarations shared between the kernel translation units and the C-ABI layer (api.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace dcr {

struct SimStats {
  int cta_group;
  int grid;
  int smem_bytes;
  int stages;
  int kp;
  int cap;
  int n_flagged;     // queries recomputed by the brute-force fp64 path
  int n_second;      // queries that needed the second-chance pass (32 candidates)
  int d_pad;
  float kernel_ms;   // device time of the fused kernel alone (CUDA events)
  float sm_mhz;      // SM clock while the fused kernel ran (clock64 / globaltimer of CTA 0; with both bias variants launched: the last one)
  int n_sets;        // epilogue warp sets of the first pass
};

size_t sim_topk_workspace_size(int nq, int ng, int d, int k);
int sim_topk(const float* q, int nq, const float* g, int ng, int d, int k, long long g_index_base,
             long long g_index_stride, float* out_scores, long long* out_idx, void* ws, size_t ws_bytes,
             cudaStream_t stream, SimStats* stats);

int split_rescore(const float* q, const float* g, int nq, int d, int n_chunks, int cross, const long long* cand, int n_cand,
                  int k, float* out_scores, long long* out_idx, cudaStream_t stream);

int l2_normalize(float* x, int n, int d, float eps, cudaStream_t stream);
// [nq, k_in] lists -> [nq, k_out >= k_in] with (-inf, -1) in the extra slots
int pad_topk_lists(const float* s_in, const long long* i_in, int nq, int k_in, int k_out, float* s_out, long long* i_out,
                   cudaStream_t stream);
int topk_merge(const float* scores, const long long* idx, int nq, int nlists, int k_in, int k_out, float* out_scores,
               long long* out_idx, cudaStream_t stream);


// ---- tcgen05 GEMM / implicit-GEMM convolution (conv_gemm.cu) ---------------------------------------------------
constexpr int kMaxGemmTerms = 6;

// Y = act(scale * conv(X, W) + bias (+ R)).  X: NHWC bf16 planes [B,H,W,C] (row stride ld_in for the 1x1/linear
// case), W: prepared weights [planes][N][kh*kw*ceil64(C)] bf16 (tap-major, channels zero-padded to 64).
struct ConvGemmDesc {
  const __nv_bfloat16* in = nullptr;
  long long in_plane_stride = 0;
  int B = 0, H = 1, W = 1, C = 0, ld_in = 0;
  // optional element strides of an overlapping-window NHWC view (0 = dense): used by the space-to-depth stem, where
  // 4 horizontally adjacent 16-channel pixels are read as one 64-channel pixel
  long long in_stride_w = 0, in_stride_h = 0, in_stride_n = 0;
  const __nv_bfloat16* weight = nullptr;
  long long w_plane_stride = 0;
  int N = 0, kh = 1, kw = 1, stride = 1, pad_h = 0, pad_w = 0;
  int n_terms = 1;
  int term_a[kMaxGemmTerms] = {0, 0, 0, 0, 0, 0};
  int term_w[kMaxGemmTerms] = {0, 0, 0, 0, 0, 0};
  const float* scale = nullptr;
  const float* bias = nullptr;
  const __nv_bfloat16* res = nullptr;
  int ld_res = 0, res_planes = 1;
  long long res_plane_stride = 0;
  __nv_bfloat16* out = nullptr;
  int ld_out = 0, out_col_off = 0, out_planes = 1;
  long long out_plane_stride = 0;
  float* out_f32 = nullptr;
  int ld_out_f32 = 0;
  int act = 0;        // 0 none, 1 relu, 2 gelu(erf)
  int exact = 0;      // 1 = float64 accumulation on the CUDA cores (conv_exact.cu) instead of the tensor cores
};
int conv_gemm(const ConvGemmDesc& d, cudaStream_t stream);
int conv_exact(const ConvGemmDesc& d, cudaStream_t stream);
bool conv3x3_halo_eligible(const ConvGemmDesc& d);   // 3x3 / stride 1 / pad 1, fast mode, no residual, W <= 62, N <= 128
int conv3x3_halo(const ConvGemmDesc& d, cudaStream_t stream);
// bottleneck_fuse.cu: `a` (1x1 expand + residual + ReLU) followed by `b` (1x1 reduce + ReLU) on a's output, fast mode
bool expand_reduce_eligible(const ConvGemmDesc& a, const ConvGemmDesc& b, size_t max_smem);
int expand_reduce(const ConvGemmDesc& a, const ConvGemmDesc& b, cudaStream_t stream);
// the same pipeline without a second convolution: K = 256 expansions with residual (ResNet-50 layer3)
bool expand_only_eligible(const ConvGemmDesc& a, size_t max_smem);
int expand_only(const ConvGemmDesc& a, cudaStream_t stream);


// ---- HBM-bound kernels (pool_norm.cu, attention.cu) ---------------------------------------------------------------
int im2col_u8(const uint8_t* img, int B, int IH, int IW, int crop_y, int crop_x, int H, int W, int kh, int kw,
              int stride, int pad, int k_pad, const float* mean3, const float* std3, float post_scale,
              float post_shift, __nv_bfloat16* out, long long out_plane_stride, int planes, cudaStream_t stream,
              const float* img_f32 = nullptr,    // img_f32: fp32 NCHW [B,3,IH,IW] already transformed (img unused)
              int RH = 0, int RW = 0, float rscale = 0.f);   // optional bilinear resize of the crop (multi_scale)
int stem_s2d_u8(const uint8_t* img, int B, int IH, int IW, int crop_y, int crop_x, int H, int W, const float* mean3,
                const float* std3, float post_scale, float post_shift, __nv_bfloat16* out, long long out_plane_stride,
                int planes, cudaStream_t stream, int RH = 0, int RW = 0, float rscale = 0.f, const float* img_f32 = nullptr);
int pool2d(bool is_max, const __nv_bfloat16* in, long long in_plane_stride, __nv_bfloat16* out,
           long long out_plane_stride, int planes, int B, int H, int W, int C, int k, int stride, int pad, int ld_out,
           int out_col_off, cudaStream_t stream);
int reduce_hw(bool gem, const __nv_bfloat16* in, long long in_plane_stride, int planes, int B, int HW, int C,
              float p_exp, float eps, __nv_bfloat16* out, long long out_plane_stride, float* out_f32,
              cudaStream_t stream);
int layernorm(const __nv_bfloat16* in, long long in_plane_stride, int planes, int rows, int C, long long in_row_stride,
              const float* gamma, const float* beta, float eps, __nv_bfloat16* out, long long out_plane_stride,
              float* out_f32, cudaStream_t stream);
int vit_tokens(const __nv_bfloat16* patch, long long patch_plane_stride, const float* cls, const float* pos,
               __nv_bfloat16* out, long long out_plane_stride, int planes, int B, int NP, int C, cudaStream_t stream);
int attention(const __nv_bfloat16* qkv, long long qkv_plane_stride, __nv_bfloat16* out, long long out_plane_stride,
              int planes, int B, int T, int heads, int dh, float scale, cudaStream_t stream, int causal = 0);
// token ids [B, T] (int32, device) -> planes[B*T, C] = table[id] + pos[t]   (CLIP text tower input, clip/model.py encode_text)
int embed_tokens(const int* ids, int B, int T, int C, const float* table, int vocab, const float* pos, __nv_bfloat16* out,
                 long long out_plane_stride, int planes, cudaStream_t stream);

// ---- fused ResNet stem (stem_fused.cu): overlapping-window (Toeplitz) A operand, fast mode ------------------------------
int stem_fused_pitch(int out_w);                              // units (16-byte pixels) per stored pair-row
long long stem_fused_plane_units(int out_h, int out_w);       // units per column-parity plane and image (incl. slack)
int stem_rows(const uint8_t* img, const float* img_f32, int B, int IH, int IW, int crop_y, int crop_x, int H, int W, int RH, int RW,
              float rscale, const float* mean3, const float* std3, float post_scale, float post_shift, __nv_bfloat16* out,
              cudaStream_t stream);
int stem_conv(const __nv_bfloat16* planes, int B, int OH, int OW, const __nv_bfloat16* weight, const float* scale, const float* bias,
              __nv_bfloat16* out, cudaStream_t stream, int pool = 0);   // pool: fuse the 3x3/2/pad-1 max pool, out = [OHp*OWp, 64]

// ---- network executor (net.cu) ------------------------------------------------------------------------------------
enum NetOpKind {
  NET_OP_IM2COL_U8 = 0,
  NET_OP_CONV = 1,
  NET_OP_MAXPOOL = 2,
  NET_OP_AVGPOOL = 3,
  NET_OP_GEM = 4,
  NET_OP_GAP = 5,
  NET_OP_LAYERNORM = 6,
  NET_OP_VIT_TOKENS = 7,
  NET_OP_ATTENTION = 8,
  NET_OP_L2NORM_OUT = 9,
  NET_OP_STEM_S2D = 10,
  NET_OP_EMBED = 11,
  NET_OP_STEM_ROWS = 12,
  NET_OP_STEM_CONV = 13,
  NET_OP_COUNT = 14
};
struct Net;
int net_create(int max_batch, int planes, Net** out);
int net_set_exact(Net* n, int on);
void net_destroy(Net* n);
int net_fork(const Net* src, Net** out);
int net_add_tensor(Net* n, long long rows_per_image, int C);
int net_alias_tensor(Net* n, int src, long long rows_per_image, int C);
int net_add_param(Net* n, const void* host, size_t bytes);
int net_set_output(Net* n, int dim);
int net_add_op(Net* n, int kind, const int* iargs, int ni, const float* fargs, int nf);
// images: uint8 NHWC [B,IH,IW,3] (raw, the transform is fused) -- or, when images_f32 != nullptr, fp32 NCHW
// [B,3,H,W] already transformed (what the reference passes to `model(samples)`, utils_ret.py:751)
int net_forward(Net* n, const uint8_t* images, int B, float* out, cudaStream_t stream, const float* images_f32 = nullptr);


// ---- FID statistics (fid.cu) ----------------------------------------------------------------------------------------
struct FidState;
int fid_create(int d, FidState** out);
void fid_destroy(FidState* s);
int fid_accumulate(FidState* s, const float* act, int n, cudaStream_t stream);
int fid_finalize(FidState* s, double* mu_host, double* sigma_host, long long* n_out, cudaStream_t stream);

}  // namespace dcr
