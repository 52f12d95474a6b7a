// kernels.cuh — launchers of the non-GEMM kernels (normalisation, operand staging, small convs,
// sampler elementwise ops, weight packing, synthetic weights).
#pragma once
#include "common.cuh"

namespace sdb {

// fp16 operand tensor [n][P][H][W][C] (hi part + optional lo residual part)
struct Half2Ptr {
  __half* hi = nullptr;
  __half* lo = nullptr;
};

// ---- GroupNorm (reference src/model/groupnorm/mod.rs:53-82), NHWC fp32, optional 2-source concat
// sums: [n][32][2] doubles (sum, sum of squares). Deterministic: per-CTA partials (scratch `partials`,
// gn_stats_partial_floats(n,HW) floats) folded in fixed order by the last CTA; `tickets` [n] must be zero.
size_t gn_stats_partial_floats(int n, int HW);
void gn_stats_launch(const float* x0, int C0, const float* x1, int C1, int n, int HW, double* sums, float* partials,
                     unsigned int* tickets, cudaStream_t st);
// One-launch GroupNorm(+SiLU) -> fp16 hi(/lo) operand: statistics and apply fused through an in-kernel grid wait.
// tickets: [n] zeroed counters; partials: gn_fused_partial_floats(n,HW) floats of scratch.
extern int g_gn_min_pix;
extern int g_gn_apply_ctas;
size_t gn_fused_partial_floats(int n, int HW);
void gn_fused_launch(const float* x0, int C0, const float* x1, int C1, int n, int H, int W, int silu, const float* gamma,
                     const float* beta, float eps, Half2Ptr out, float* partials, unsigned int* tickets, cudaStream_t st);
// GroupNorm(+SiLU) -> fp16 hi(/lo) operand from statistics the producing GEMM left beside the tensor (gemm_tc.cuh: gn_part):
// one read of x, no statistics pass, no rendezvous. part = [n][cap][C / bucket][2] floats, `slots` of the cap written.
struct GnSrc {
  const float* x = nullptr;
  int C = 0;
  const float* part = nullptr;
  int cap = 0, slots = 0;
};
// folds groups of 64 partial slots: out [n][gn_fold_slots(slots)][nbk][2]
int gn_fold_slots(int slots);
void gn_fold_launch(const float* part, int cap, int slots, int nbk, int n, float* out, cudaStream_t st);
// group sums [n][32][2] of one tensor from its producer-side partials (cap / slots as in GnSrc)
void gn_sums_from_partials_launch(const float* part, int cap, int slots, int nbk, int C, int bucket, int n, double* sums,
                                  cudaStream_t st);
void gn_apply_launch(const GnSrc& s0, const GnSrc& s1, int bucket, int n, int H, int W, int silu, const float* gamma,
                     const float* beta, float eps, Half2Ptr out, cudaStream_t st);
// mode bits
enum : int { PREP_NORM = 1, PREP_SILU = 2, PREP_UP2 = 4, PREP_PHASE2 = 8 };
// Stages a conv/GEMM A operand: y = [silu]([groupnorm](cat(x0,x1))) -> fp16 hi(/lo).
//   PREP_UP2    : nearest 2x upsample while writing (output [n][2H][2W][C])
//   PREP_PHASE2 : split into 4 stride-2 phase planes (output [n][4][H/2][W/2][C])
void prep_operand_launch(const float* x0, int C0, const float* x1, int C1, int n, int H, int W, int mode,
                         const double* sums, const float* gamma, const float* beta, float eps, Half2Ptr out,
                         cudaStream_t st);
// fp32 output variant of GroupNorm(+SiLU) used by the unit-test entry and by the small-N convs
void gn_apply_f32_launch(const float* x, int C, int n, int HW, int silu, const double* sums, const float* gamma,
                         const float* beta, float eps, float* y, cudaStream_t st);

// ---- LayerNorm (burn nn::LayerNorm; call sites unet/mod.rs:523-525): rows x C fp32 -> fp16 hi(/lo) or fp32
void layernorm_launch(const float* x, int rows, int C, const float* gamma, const float* beta, float eps,
                      Half2Ptr out, float* out_f32, cudaStream_t st);

// ---- plain fp32 -> fp16 hi(/lo) conversion (context tokens, test inputs)
void convert_f16_launch(const float* x, long long count, Half2Ptr out, cudaStream_t st);

// ---- layout conversion at the boundary
void nchw_to_nhwc_launch(const float* x, int n, int C, int H, int W, float* y, cudaStream_t st);
void nhwc_to_nchw_launch(const float* x, int n, int C, int H, int W, float* y, cudaStream_t st);

// ---- small convolutions on CUDA cores (fp32 exact)
// 3x3 pad 1, Cin = 4 (NCHW fp32 input [n,4,H,W]) -> NHWC fp32 [n,H,W,Cout]; weights OIHW fp32.
// pre: optional 1x1 4->4 conv (post_quant_conv) with scalar input scale applied to the input first.
void conv3x3_cin4_launch(const float* x_nchw, int n, int H, int W, const float* w, const float* b, int Cout,
                         const float* pre_w, const float* pre_b, float pre_scale, float* y, Half2Ptr y16, cudaStream_t st);
// 3x3 pad 1, Cout <= 4, input NHWC fp32 with fused GroupNorm+SiLU; output NCHW fp32 [n,Cout,H,W];
// weights repacked [Cout][9][C] fp32.
void conv3x3_small_cout_launch(const float* x, int n, int H, int W, int C, const double* sums, const float* gamma,
                               const float* beta, float eps, const float* w_packed, const float* b, int Cout,
                               float* y_nchw, cudaStream_t st);

// ---- time embedding (reference unet/mod.rs:19-30, 115-118, 718-722)
// emb = lin2(silu(lin1([cos|sin](t*f)))) ; then for every ResBlock r: e_r = lin_embed_r(silu(emb))
void time_embed_launch(const int* t_dev, const float* w1, const float* b1, const float* w2, const float* b2, float* hidden,
                       float* emb_silu, cudaStream_t st);
// the same for `rows` timesteps at once (t_dev[rows]); emb_all[t][n_all] is indexed by the timestep value. Bit-identical rows.
void time_embed_rows_launch(const int* t_dev, int rows, const float* w1, const float* b1, const float* w2, const float* b2,
                            const float* w_all, const float* b_all, int n_all, float* hidden, float* emb_silu, float* emb_all,
                            cudaStream_t st);
void emb_select_launch(const float* emb_all, const int* t_dev, int N, float* out, cudaStream_t st);
// y[N] = x[K] @ W[K][N] + b  (tiny GEMV, W fp32 [in,out])
void gemv_launch(const float* x, const float* W, const float* b, int K, int N, float* y, cudaStream_t st);

// ---- CLIP embedding lookup: x [n][Lp][D] = E[tok] + Pos, rows l >= L zero (reference clip/mod.rs:62-68)
void embed_tokens_launch(const int* tok, const float* E, const float* Pos, int n, int L, int Lp, int D, int vocab, float* x,
                         cudaStream_t st);

// ---- sampler elementwise (reference stablediffusion/mod.rs:152-156, 190-191)
// pred = u + (c-u)*scale ; x0 = (lat - pred*sqrt(1-a_t))/sqrt(a_t) ; lat' = x0*sqrt(a_prev) + pred*sqrt(1-a_prev)
// latent holds 2*count floats: the update is written to both halves (uncond | cond inputs of the next step)
void cfg_ddim_launch(const float* eps_u, const float* eps_c, float* latent, long long count, float scale,
                     float sqrt_one_minus_at, float sqrt_at, float sqrt_aprev, float dir_coef, cudaStream_t st);
// pred = u + (c - u) * scale alone (forward_diffuser without the DDIM update)
void cfg_combine_launch(const float* eps_u, const float* eps_c, long long count, float scale, float* pred, cudaStream_t st);
// u8 = trunc(clamp((img+1)/2*255, 0, 255)), NCHW fp32 -> NHWC u8 (reference stablediffusion/mod.rs:79-97)
void to_rgb8_launch(const float* img_nchw, int n, int H, int W, uint8_t* rgb, cudaStream_t st);
// ---- img2img / inpainting (DESIGN.md §7 row f5)
// u8 HWC [n][H][W][3] -> fp32 NCHW [n][4][H][W] with a zero fourth plane: x = fl(fl(v * fl32(2/255)) - 1), no FMA
void rgb8_to_planes4_launch(const uint8_t* rgb, int n, int H, int W, float* img4, cudaStream_t st);
// pixel mask [n][8H][8W] (nonzero = repaint) -> latent mask [n][H][W] in {0,1}: max over each 8x8 block
void latent_mask_launch(const uint8_t* mask, int n, int H, int W, uint8_t* m, cudaStream_t st);
// x = fl(x * s) in place
void scale_launch(float* x, long long count, float s, cudaStream_t st);
// x_t0 = fl(fl(a*x0) + fl(b*eps)), written to both halves of latent [2*count] (uncond | cond inputs)
void noise_latent_launch(const float* x0, const float* eps, long long count, float a, float b, float* latent, cudaStream_t st);
// cfg_ddim_launch, then cells with m[n][HW] == 0 take fl(fl(sqrt_aprev*x0) + fl(dir_coef*eps)); latent [n][4][HW] twice
void cfg_ddim_blend_launch(const float* eps_u, const float* eps_c, float* latent, long long count, float scale,
                           float sqrt_one_minus_at, float sqrt_at, float sqrt_aprev, float dir_coef, const float* x0,
                           const float* eps, const uint8_t* m, int HW, cudaStream_t st);
// to_rgb8_launch where pixels with mask[n][H][W] == 0 are copied from src_rgb [n][H][W][3]
void to_rgb8_paste_launch(const float* img_nchw, int n, int H, int W, const uint8_t* src_rgb, const uint8_t* mask, uint8_t* rgb,
                          cudaStream_t st);
void quant_conv_slice_launch(const float* x, const float* w, const float* b, int n, int HW, float* y, cudaStream_t st);
void add_vec_launch(const float* a, const float* b, int n, float* y, cudaStream_t st);
// N(0,1) latents from a Philox-like counter hash (used only when the caller passes no init latent)
void randn_launch(float* x, long long count, uint64_t seed, cudaStream_t st);
// ---- selectable samplers (DESIGN.md §7 row f6): CFG + update in one launch, one rounding per operation (no contraction)
// DDIM with eta > 0: lat' = x0*sqrt_anext + pred*dir + sigma*z; z = z[i], or randn_launch(z_seed)'s element i drawn in-kernel
// when z is null; sigma == 0 reads no noise. latent holds 2*count floats, written to both halves like cfg_ddim_launch.
void cfg_ddim_eta_launch(const float* eps_u, const float* eps_c, float* latent, long long count, float scale,
                         float sqrt_one_minus_at, float sqrt_at, float sqrt_anext, float dir, float sigma, const float* z,
                         uint64_t z_seed, cudaStream_t st);
// DPM-Solver++(2M), kind 0 = first order, 1 = second order, 2 = final (lat' = x0): D = x0 | x0*w0 - hist*w1,
// lat' = x*ratio - D*coef; hist [count] = x0 of the previous step, overwritten with this step's (kinds 0 and 1 only)
void cfg_dpmpp2m_launch(int kind, const float* eps_u, const float* eps_c, float* latent, float* hist, long long count, float scale,
                        float sqrt_one_minus_at, float sqrt_at, float ratio, float coef, float w0, float w1, cudaStream_t st);

// ---- row softmax for the 1-head VAE attention: P = softmax(S*scale) rows -> fp16 hi(/lo)
void softmax_rows_launch(const float* S, long long rows, int cols, float scale, Half2Ptr out, cudaStream_t st);

// ---- weight packing (master fp32 -> kernel layouts)
// conv OIHW [Cout][Cin][k][k] -> [Cout][k*k*Cin] with K index = tap*Cin + c ; fp16 hi (+lo)
void pack_conv_launch(const float* w, int Cout, int Cin, int ksize, Half2Ptr out, cudaStream_t st);
// nearest-2x-upsample folded 3x3 conv: 4 output phases x 2x2 taps, [4][Cout][4*Cin]
void pack_conv_up2_launch(const float* w, int Cout, int Cin, Half2Ptr out, cudaStream_t st);
// Linear [in][out] -> [out_row_offset + out][in] inside a packed matrix of row length ld (=in)
// ldw/col0 select a column slice [col0, col0+out) of a source matrix with row stride ldw (0 -> out)
// in_scale (optional, [in]): multiplies input feature i — a LayerNorm gamma folded into the consuming GEMM's weights
void pack_linear_launch(const float* w, int in, int out, Half2Ptr dst, int row_offset, cudaStream_t st, int ldw = 0,
                        int col0 = 0, const float* in_scale = nullptr);
// per-row sums of a packed fp16 matrix [rows][K]: s_hi = sum hi, s_full = sum (hi + lo); either output may be null
void rowsum_f16_launch(Half2Ptr m, int rows, int K, float* s_hi, float* s_full, cudaStream_t st);
// GEGLU proj [in][2*H4] -> rows interleaved per 2*half-tile: tile j holds x rows j*half.. then gate rows
void pack_geglu_launch(const float* w, const float* b, int in, int h4, int half_tile, Half2Ptr dst, float* bias_packed,
                       cudaStream_t st, const float* in_scale = nullptr);
// conv OIHW (Cout<=4, 3x3) -> fp32 [Cout][9][Cin]
void pack_small_cout_launch(const float* w, int Cout, int Cin, float* out, cudaStream_t st);

// ---- synthetic weights (bit-identical to stable_diffusion_burn_b200/synth.py)
void synth_fill_launch(float* dst, long long count, uint32_t key, float bound, float offset, cudaStream_t st);
struct SynthDesc {
  long long offset, count, chunk0;  // float offset in the arena, element count, index of the tensor's first 64K-element chunk
  uint32_t key;
  float bound, shift;
};
void synth_fill_table_launch(float* base, const SynthDesc* d_desc, int ntensors, long long nchunks, cudaStream_t st);

}  // namespace sdb
