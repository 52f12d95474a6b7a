/*
 * sdb200.h — C ABI of the B200-native Stable Diffusion v1.4 sampling path.
 *
 * Drop-in boundary for the hot path of Gadersd/stable-diffusion-burn (reference @ 893fb095):
 * these entry points are what a Rust FFI shim binds in place of the Burn tensor graph in
 * src/backend.rs and src/model/{unet,attention,groupnorm,autoencoder}. Each function cites the
 * reference interface it replaces. The reference-side binding is shown in INTEGRATION.md and
 * rust/sdb200_ffi.rs.
 *
 * Conventions
 *  - every call returns int: 0 = ok, non-zero = error (text via sdb_last_error); nothing
 *    unwinds across the boundary (the reference panics / exit(1)s: src/bin/sample/main.rs:45-52).
 *  - tensors are contiguous row-major fp32, NCHW / [n, seq, C], exactly the reference's
 *    Tensor<B,4> / Tensor<B,3> contents. Caller owns every buffer; the library owns the context.
 *  - host-pointer calls are synchronous on return. *_dev variants take device pointers and a
 *    cudaStream_t (passed as void*) and are asynchronous on that stream.
 *  - a context is bound to one CUDA device and is not re-entrant (one in-flight call per ctx).
 *  - there is NO CPU fallback: every compute entry fails if the device path is unavailable.
 */
#ifndef SDB200_H
#define SDB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sdb_ctx sdb_ctx;

/* ---- lifetime ------------------------------------------------------------------------- */
/* Replaces device selection + StableDiffusionConfig::init (src/bin/sample/main.rs:59-83,
 * src/model/stablediffusion/mod.rs:22-39). */
int sdb_create(int device, sdb_ctx** out);
int sdb_destroy(sdb_ctx* ctx);
/* ctx may be NULL: returns the last error of the calling thread (e.g. a failed sdb_create). */
const char* sdb_last_error(sdb_ctx* ctx);
/* "sdb200 <version> sm_100a" */
const char* sdb_version(void);

/* ---- weights -------------------------------------------------------------------------- */
/* Tensor registry. Names are the reference's dump-dir paths (src/model/unet/load.rs:213-306,
 * src/model/autoencoder/load.rs:16-198), e.g. "unet/input_blocks/rt1/res/conv_in/weight";
 * Linear weights are [in,out] and conv weights OIHW as in src/model/load.rs:65-160. The extra
 * tensor "alpha_cumulative_products" [1000] is the sampler's schedule Param
 * (src/model/stablediffusion/mod.rs:44). */
int sdb_tensor_count(sdb_ctx* ctx);
int sdb_tensor_info(sdb_ctx* ctx, int index, const char** name, int64_t dims[4], int* ndim);
/* Replaces load_tensor -> Param::from_tensor (src/model/load.rs:30-47). host: fp32, dims must match. */
int sdb_set_tensor(sdb_ctx* ctx, const char* name, const float* host, const int64_t* dims, int ndim);
/* Reads back the fp32 master copy (tests / checkpoint round trips). */
int sdb_get_tensor(sdb_ctx* ctx, const char* name, float* host, int64_t count);
/* load_stable_diffusion (src/model/stablediffusion/load.rs:16-33) for the part of the model on this path: reads every
 * registry tensor from the reference's dump-dir tree (1-D f32 .npy = [dims..., values...], python/save.py:10-15 <->
 * src/model/load.rs:17-47; <path>/<tensor name>.npy, the schedule from <path>/alphas_cumprod.npy). Optional files follow
 * the reference (missing Linear/Conv bias = none, missing GroupNorm weight/bias = ones/zeros); the configuration scalars
 * the reference reads (eps, n_group, stride, padding, n_head, n_layer, n_steps ...) are validated against the compiled
 * SD-v1.4 topology and each norm's eps is honoured. The encoder / quant_conv files are read too (sdb_encode_image and
 * sdb_img2img use them). */
int sdb_load_dump_dir(sdb_ctx* ctx, const char* path);
/* load_tensor::<B, D> (src/model/load.rs:30-47) for one file, no context needed: splits the leading `ndim` shape values
 * from the data. Returns the element count (data may be NULL to probe), or -1 (text via sdb_last_error(NULL)). */
int64_t sdb_read_dump_tensor(const char* file, int ndim, int64_t* dims, float* data, int64_t capacity);
/* Fills every tensor with the deterministic synthetic stream documented in
 * stable_diffusion_burn_b200/synth.py (bit-identical to the numpy generator). */
int sdb_init_synthetic(sdb_ctx* ctx, uint32_t seed);
/* fp32 master arena (device pointer, bytes): one contiguous block holding every tensor, for the
 * single init-time ncclBroadcast from rank 0 (SURVEY §8e). */
int sdb_weight_arena(sdb_ctx* ctx, void** dev_ptr, size_t* bytes);
/* Multi-GPU init (SURVEY §8b(2), §8e): the ONE collective of the path. Rank 0 obtains an id with sdb_nccl_unique_id (128 bytes,
 * = ncclUniqueId) and hands it to every rank by its own means (file, socket, MPI, torch store); then every rank calls
 * sdb_broadcast_weights(ctx, id, rank, world): ncclCommInitRank + ncclBroadcast of the fp32 master arena (and of the per-norm
 * eps table a dump-dir carries) from rank 0 over NVLink, then the communicator is destroyed — no collective on the sampling
 * path. NCCL is resolved with dlopen("libnccl.so.2") at the first call: single-GPU hosts need no NCCL. world == 1 is a no-op.
 * Call sdb_finalize_weights afterwards on every rank. */
int sdb_nccl_unique_id(void* id128);
int sdb_broadcast_weights(sdb_ctx* ctx, const void* id128, int rank, int world);
/* Packs the master weights into kernel layouts (fp16 K-major tiles, fused QKV/GEGLU orders).
 * Must be called after the last sdb_set_tensor / broadcast and before any compute call. */
int sdb_finalize_weights(sdb_ctx* ctx);

/* ---- hot path, host buffers -------------------------------------------------------------- */
/* UNet::forward (src/model/unet/mod.rs:109-142): x [n,4,H,W], one timestep for the batch,
 * context [n,L,768] -> out [n,4,H,W]. */
int sdb_unet_forward(sdb_ctx* ctx, const float* x, int32_t timestep, const float* context,
                     int n, int H, int W, int L, float* out);
/* Autoencoder::decode_latent (src/model/autoencoder/mod.rs:68-71): latent [n,4,H,W] -> img [n,3,8H,8W]. */
int sdb_decode_latent(sdb_ctx* ctx, const float* latent, int n, int H, int W, float* img);
/* StableDiffusion::sample_latent (src/model/stablediffusion/mod.rs:102-160), DDIM eta=0 with
 * classifier-free guidance (forward_diffuser :162-192). context [n,L,768]; uncond [Lu,768] is
 * broadcast over the batch. init_latent [n,4,H,W] (the reference draws it from an unseeded RNG,
 * :115-121); if NULL an internal Philox N(0,1) stream keyed by `seed` is used. */
int sdb_sample_latent(sdb_ctx* ctx, const float* context, int n, int L, const float* uncond, int Lu,
                      double guidance_scale, int n_steps, const float* init_latent, uint64_t seed,
                      int H, int W, float* latent_out);
/* StableDiffusion::forward_diffuser (src/model/stablediffusion/mod.rs:162-192): classifier-free guidance at one timestep,
 * pred = u + (c - u) * scale with u = UNet(latent, t, uncond broadcast over the batch), c = UNet(latent, t, context) — evaluated
 * as ONE batch-2n UNet pass (the pass sample_latent replays per step). latent [n,4,H,W]; pred / out_uncond / out_cond [n,4,H,W],
 * each may be NULL (out_uncond / out_cond expose the two UNet outputs before the combine, for per-step parity checks). */
int sdb_forward_diffuser(sdb_ctx* ctx, const float* latent, int32_t timestep, const float* context, int n, int L,
                         const float* uncond, int Lu, double guidance_scale, int H, int W, float* pred,
                         float* out_uncond, float* out_cond);
/* StableDiffusion::latent_to_image (src/model/stablediffusion/mod.rs:69-100): decode(latent/0.18215),
 * (x+1)/2*255, NHWC, clamp to [0,255], truncate to u8. rgb [n,8H,8W,3]. */
int sdb_latent_to_image(sdb_ctx* ctx, const float* latent, int n, int H, int W, uint8_t* rgb);
/* StableDiffusion::sample_image (src/model/stablediffusion/mod.rs:51-67) = sample_latent + latent_to_image. */
int sdb_sample_image(sdb_ctx* ctx, const float* context, int n, int L, const float* uncond, int Lu,
                     double guidance_scale, int n_steps, const float* init_latent, uint64_t seed,
                     int H, int W, uint8_t* rgb);

/* ---- text encoder (SURVEY §8f row f1: the first "next" row after the hot path) ------------------ */
/* CLIP::forward (src/model/clip/mod.rs:56-75): token ids [n,L] (L <= 77, NOT padded — the reference does not pad,
 * src/model/stablediffusion/mod.rs:198-211) -> context [n,L,768]. The ids come from SimpleTokenizer::encode
 * (src/tokenizer.rs:175-195), mirrored host-side in stable_diffusion_burn_b200/tokenizer.py. */
int sdb_clip_forward(sdb_ctx* ctx, const int32_t* tokens, int n, int L, float* out);
/* device-pointer variant: ids outside [0,49408) are clamped (the host variant rejects them). */
int sdb_clip_forward_dev(sdb_ctx* ctx, const int32_t* d_tokens, int n, int L, float* d_out, void* stream);

/* ---- VAE encoder (SURVEY §8f row f4) ---------------------------------------------------------------- */
/* Autoencoder::encode_image (src/model/autoencoder/mod.rs:60-66): img [n,3,H,W] -> latent [n,4,H/8,W/8] = the first four
 * channels of quant_conv(encoder(img)). H, W multiples of 8 (>= 64). sdb_img2img builds on it; the reference CLI never calls it. */
int sdb_encode_image(sdb_ctx* ctx, const float* img, int n, int H, int W, float* latent);
int sdb_encode_image_dev(sdb_ctx* ctx, const float* d_img, int n, int H, int W, float* d_latent, void* stream);

/* ---- img2img and inpainting (DESIGN.md §7 row f5) ------------------------------------------------------- */
/* The reference has no img2img; this is SDEdit / latent-blend inpainting on its schedule and sampler
 * (src/model/stablediffusion/mod.rs:102-160). H, W are latent sizes as in sdb_sample_image.
 *  rgb [n,8H,8W,3] u8 (the layout sdb_sample_image writes) -> x = rgb * fl32(2/255) - 1 -> x0 = 0.18215 * encode_image(x).
 *  Of the T timesteps of the n_steps schedule the last n_run = min(T, floor(strength * T + 1e-9)) run, starting from
 *  sqrt(a[t0]) x0 + sqrt(1 - a[t0]) noise; strength 0 returns x0 with no UNet pass. noise [n,4,H,W], or NULL for the N(0,1)
 *  stream keyed by `seed` that sdb_sample_latent draws its initial latent from.
 *  mask [n,8H,8W] u8 or NULL: nonzero = repaint. A latent cell is repainted if any pixel of its 8x8 block is; after every
 *  step the other cells are reset to the known image noised to the step's target timestep (x0 itself after the last step),
 *  and rgb_out pixels whose mask is 0 are copied from rgb. The SD-v1.4 UNet has 4 input channels: no 9-channel inpainting.
 *  latent_out [n,4,H,W] and rgb_out [n,8H,8W,3] may each be NULL, but not both. Errors: strength NaN or outside [0,1],
 *  rgb NULL, n_steps outside [1,1000], sizes the encoder or the UNet reject. */
int sdb_img2img(sdb_ctx* ctx, const uint8_t* rgb, const uint8_t* mask, const float* context, int n, int L,
                const float* uncond, int Lu, double guidance_scale, int n_steps, double strength,
                const float* noise, uint64_t seed, int H, int W, float* latent_out, uint8_t* rgb_out);
int sdb_img2img_dev(sdb_ctx* ctx, const uint8_t* d_rgb, const uint8_t* d_mask, const float* d_context, int n, int L,
                    const float* d_uncond, int Lu, double guidance_scale, int n_steps, double strength,
                    const float* d_noise, uint64_t seed, int H, int W, float* d_latent_out, uint8_t* d_rgb_out,
                    void* stream);

/* ---- selectable samplers (DESIGN.md §7 row f6) ----------------------------------------------------------- */
/* The reference's only sampler is DDIM with sigma fixed to 0 (src/model/stablediffusion/mod.rs:119; the noise term at :155
 * never runs). sdb_sample_ex runs sample_latent's loop (:102-160) with a selectable update on the same schedule
 * (ts = (0..1000).rev().step_by(1000 / n_steps), T = len(ts), a_next = 1 after the last step):
 *  SDB_SAMPLER_DDIM, eta in [0,1]: x' = x0 sqrt(a_next) + pred sqrt(1 - a_next - sigma^2) + sigma z_i with
 *    sigma = eta sqrt((1 - a_next)/(1 - a_t)) sqrt(1 - a_t/a_next) (0 at the last step). eta = 0 is sdb_sample_latent exactly.
 *  SDB_SAMPLER_DPMPP_2M (eta = 0): DPM-Solver++(2M), data prediction; first order at step 0, second order after it, and the
 *    last step returns its x0 prediction.
 * step_noise [T][n,4,H,W]: z_i is slice i; the last slice must be present but is never read (sigma = 0 there). Given only for
 * DDIM with eta > 0. NULL: slice i is sdb_randn(seed_i, n*4*H*W) with seed_i = seed ^ ((i+1) * 0x9E3779B97F4A7C15) mod 2^64,
 * drawn inside the update kernel. init_latent NULL: sdb_randn(seed, n*4*H*W), as sdb_sample_latent.
 * latent_out [n,4,H,W] and rgb_out [n,8H,8W,3] may each be NULL, but not both. Errors: unknown sampler, eta NaN or outside
 * [0,1], eta != 0 with DPM-Solver++(2M), step_noise with any other sampler than DDIM at eta > 0, and what sdb_sample_latent
 * rejects. The time-embedding hoist and the cached step graph of sdb_sample_latent are used unchanged. */
#define SDB_SAMPLER_DDIM 0     /* eta >= 0; eta = 0 is sdb_sample_latent exactly */
#define SDB_SAMPLER_DPMPP_2M 1
int sdb_sample_ex(sdb_ctx* ctx, const float* context, int n, int L, const float* uncond, int Lu, double guidance_scale,
                  int n_steps, int sampler, double eta, const float* init_latent, const float* step_noise, uint64_t seed,
                  int H, int W, float* latent_out, uint8_t* rgb_out);
int sdb_sample_ex_dev(sdb_ctx* ctx, const float* d_context, int n, int L, const float* d_uncond, int Lu, double guidance_scale,
                      int n_steps, int sampler, double eta, const float* d_init_latent, const float* d_step_noise, uint64_t seed,
                      int H, int W, float* d_latent_out, uint8_t* d_rgb_out, void* stream);
/* The library's seeded N(0,1) stream (the initial latent of sdb_sample_latent / sdb_sample_ex and the step noise above):
 * count values into host memory. */
int sdb_randn(sdb_ctx* ctx, uint64_t seed, int64_t count, float* out);

/* ---- hot path, device buffers (zero-copy callers) ------------------------------------------ */
int sdb_unet_forward_dev(sdb_ctx* ctx, const float* d_x, int32_t timestep, const float* d_context,
                         int n, int H, int W, int L, float* d_out, void* stream);
int sdb_decode_latent_dev(sdb_ctx* ctx, const float* d_latent, int n, int H, int W, float* d_img, void* stream);
int sdb_forward_diffuser_dev(sdb_ctx* ctx, const float* d_latent, int32_t timestep, const float* d_context, int n, int L,
                             const float* d_uncond, int Lu, double guidance_scale, int H, int W, float* d_pred, void* stream);
int sdb_sample_image_dev(sdb_ctx* ctx, const float* d_context, int n, int L, const float* d_uncond, int Lu,
                         double guidance_scale, int n_steps, const float* d_init_latent,
                         int H, int W, uint8_t* d_rgb, void* stream);

/* ---- configuration / instrumentation ------------------------------------------------------- */
/* key/value knobs: "precision" = 1|2|3 tensor-core passes per product (0 = the per-layer policy, see DESIGN.md),
 * "graphs" = 0|1 (CUDA-graph replay of the UNet step), "splitk" = 0|1. A/B switches of measured design choices (defaults are the
 * measured-faster settings; results do not change beyond rounding, the first two not at all): "emb_hoist" (time-embedding rows of
 * all timesteps once per sample call), "attn_regsplit" (setmaxnreg build of the attention kernel), "attn_split" (fp16 hi + lo
 * q / k on the 3-pass levels), "prefetch_w", "cluster", "pair_bn256", "raw16", "skip_merge", "gn_epilogue", "mlp_passes",
 * "splitk_min_iters", "splitk_chunk", "gn_apply_ctas", "gn_min_pix". Unknown keys are an error. */
int sdb_set_option(sdb_ctx* ctx, const char* key, int value);
/* Per-kernel-class timing: when enabled, every launch is bracketed by CUDA events on the
 * context's stream (graphs are bypassed). */
int sdb_profile_enable(sdb_ctx* ctx, int on);
int sdb_profile_reset(sdb_ctx* ctx);
int sdb_profile_class_count(sdb_ctx* ctx);
/* launches, total device milliseconds, algorithmic FLOPs and bytes of one kernel class. */
int sdb_profile_get(sdb_ctx* ctx, int cls, const char** name, int64_t* launches, double* ms,
                    double* flops, double* bytes);
/* tensor-core FLOPs actually issued by a class (x2 / x3 of the algorithmic count where the split-fp16 product runs). */
int sdb_profile_get_issued(sdb_ctx* ctx, int cls, double* issued_flops);
/* Number of kernel launches issued by this context since creation (sdb_profile_reset zeroes it). */
int64_t sdb_launch_count(sdb_ctx* ctx);

/* ---- unit-test entry points for single kernels (device pointers) ----------------------------- */
/* C[M,N] (fp32) = A[M,K] (fp32, rounded to the operand format) x B[K,N] (fp32 [in,out]) + bias.
 * Exercises the tcgen05 GEMM exactly as the Linear layers use it. */
int sdb_test_linear(sdb_ctx* ctx, const float* a, const float* w, const float* bias, int M, int K, int N,
                    int passes, float* c);
/* The GEMM's other epilogues and K-loop forms, each reachable in isolation: out = A[M,K] x W[K,N] (+ bias) (+ residual[M,N])
 * (+ XA[M,XK] x XW[XK,N], the "extra K" operands the ResBlock skip conv rides on). flags: 1 = GEGLU (W = [K][x | gate], out
 * [M, N/2] = (x + b_x) * gelu_erf(gate + b_g), unet/mod.rs:578-592); 4 = read the result back from the fp16 hi + lo outputs.
 * Split-K is chosen by the library's own policy (small M x N grid, K >= 2048). */
int sdb_test_gemm_ex(sdb_ctx* ctx, const float* a, const float* w, const float* bias, const float* residual, int M, int K,
                     int N, int passes, int flags, const float* xa, const float* xw, int XK, float* out);
/* conv2d NCHW fp32 in/out through the implicit-GEMM path (3x3 pad 1 stride 1|2, or 1x1). */
int sdb_test_conv2d(sdb_ctx* ctx, const float* x, const float* w, const float* bias, int n, int cin, int H,
                    int W, int cout, int ksize, int stride, int upsample, int passes, float* y);
/* The LayerNorm-free TransformerBlock chain in isolation (unet/mod.rs:521-527): y = a w0 + b0 (+ a2 w0 + b0 accumulated in place
 * on the fp16 hi/lo residual pair; a2 may be NULL) with row statistics from the producing epilogue, then
 * out = LayerNorm(y; gamma, beta) w1 + b1 with the LayerNorm folded into the consuming GEMM (gamma in the weights, rank-1
 * correction in the epilogue); geglu = 1: w1 = [C][x | gate], out [M, N/2] = x * gelu(gate). C a multiple of 160. */
int sdb_test_ln_fold(sdb_ctx* ctx, const float* a, const float* a2, const float* w0, const float* b0, const float* gamma,
                     const float* beta, const float* w1, const float* b1, int M, int K0, int C, int N, int passes, int geglu,
                     float* out);
/* conv (3x3 pad 1 or 1x1) whose epilogue also leaves the GroupNorm statistics of its output, followed by the apply-only
 * GroupNorm(+SiLU) that consumes them (the ResBlock's conv_in -> norm_out -> SiLU chain, unet/mod.rs:716-725). NCHW fp32 in/out;
 * *slots = partial-statistics slots per image the GEMM wrote (> 0). */
int sdb_test_conv_groupnorm(sdb_ctx* ctx, const float* x, const float* w, const float* bias, const float* gamma,
                            const float* beta, int n, int cin, int H, int W, int cout, int ksize, int passes, int silu,
                            float* y, int* slots);
/* GroupNorm(32 groups)+optional SiLU, NCHW fp32 in/out. */
int sdb_test_groupnorm(sdb_ctx* ctx, const float* x, const float* gamma, const float* beta, int n, int c,
                       int H, int W, int silu, float* y);
/* LayerNorm over the last dim, [rows, c]. */
int sdb_test_layernorm(sdb_ctx* ctx, const float* x, const float* gamma, const float* beta, int rows, int c,
                       float* y);
/* qkv_attention (src/model/attention.rs:5-45): q [n,Nq,C], k,v [n,Nk,C], heads -> out [n,Nq,C]. */
int sdb_test_attention(sdb_ctx* ctx, const float* q, const float* k, const float* v, int n, int Nq, int Nk,
                       int C, int heads, float* out);

#ifdef __cplusplus
}
#endif
#endif /* SDB200_H */
