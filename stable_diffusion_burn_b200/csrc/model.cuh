// model.cuh — the SD-v1.4 sampling graph on top of the kernels (UNet, VAE decoder, DDIM sampler).
#pragma once
#include "runtime.cuh"

namespace sdb {

void model_create(Ctx& c);   // builds the tensor registry, allocates arenas
void model_destroy(Ctx& c);
void model_init_synthetic(Ctx& c, uint32_t seed);
void model_finalize(Ctx& c);  // packs weights into kernel layouts
void model_invalidate_graphs(Ctx& c);

void model_unet_forward_host(Ctx& c, const float* x, int t, const float* context, int n, int H, int W, int L, float* out);
void model_unet_forward_dev(Ctx& c, const float* d_x, int t, const float* d_context, int n, int H, int W, int L,
                            float* d_out, cudaStream_t caller);
void model_decode_host(Ctx& c, const float* latent, int n, int H, int W, float* img);
void model_decode_dev(Ctx& c, const float* d_latent, int n, int H, int W, float* d_img, cudaStream_t caller);
void model_encode_host(Ctx& c, const float* img, int n, int H, int W, float* latent);
void model_encode_dev(Ctx& c, const float* d_img, int n, int H, int W, float* d_latent, cudaStream_t caller);
void model_latent_to_image_host(Ctx& c, const float* latent, int n, int H, int W, uint8_t* rgb);
void model_sample_host(Ctx& c, const float* context, int n, int L, const float* uncond, int Lu, double scale, int n_steps,
                       const float* init_latent, uint64_t seed, int H, int W, float* latent_out, uint8_t* rgb);
void model_sample_dev(Ctx& c, const float* d_context, int n, int L, const float* d_uncond, int Lu, double scale,
                      int n_steps, const float* d_init_latent, int H, int W, float* d_latent_out, uint8_t* d_rgb,
                      cudaStream_t caller);
// img2img / latent-blend inpainting on the DDIM sampler: rgb [n,8H,8W,3] u8, optional pixel mask [n,8H,8W] (nonzero =
// repaint), optional noise [n,4,H,W] (else randn_launch keyed by seed); latent_out / rgb_out may each be null, not both
void model_img2img_dev(Ctx& c, const uint8_t* d_rgb_in, const uint8_t* d_mask, const float* d_context, int n, int L,
                       const float* d_uncond, int Lu, double scale, int n_steps, double strength, const float* d_noise,
                       uint64_t seed, int H, int W, float* d_latent_out, uint8_t* d_rgb, cudaStream_t caller);
void model_img2img_host(Ctx& c, const uint8_t* rgb_in, const uint8_t* mask, const float* context, int n, int L,
                        const float* uncond, int Lu, double scale, int n_steps, double strength, const float* noise, uint64_t seed,
                        int H, int W, float* latent_out, uint8_t* rgb);
// text-to-image with a selectable sampler (DESIGN.md §7 row f6): sampler SAMPLER_DDIM (eta in [0,1]; eta = 0 is
// model_sample_dev exactly) or SAMPLER_DPMPP_2M (eta = 0). step_noise [T][n,4,H,W] (DDIM with eta > 0 only) or null: slice i is
// then drawn in-kernel from the randn_launch stream keyed by sampler_step_seed(seed, i). init_latent null: randn_launch(seed).
enum SamplerKind : int { SAMPLER_DDIM = 0, SAMPLER_DPMPP_2M = 1 };
uint64_t sampler_step_seed(uint64_t seed, int i);
void model_sample_ex_dev(Ctx& c, const float* d_context, int n, int L, const float* d_uncond, int Lu, double scale, int n_steps,
                         int sampler, double eta, const float* d_init_latent, const float* d_step_noise, uint64_t seed, int H, int W,
                         float* d_latent_out, uint8_t* d_rgb, cudaStream_t caller);
void model_sample_ex_host(Ctx& c, const float* context, int n, int L, const float* uncond, int Lu, double scale, int n_steps,
                          int sampler, double eta, const float* init_latent, const float* step_noise, uint64_t seed, int H, int W,
                          float* latent_out, uint8_t* rgb);
// the N(0,1) stream of randn_launch keyed by seed, count values into host memory
void model_randn_host(Ctx& c, uint64_t seed, int64_t count, float* out);
void model_forward_diffuser_dev(Ctx& c, const float* d_latent, int t, const float* d_context, int n, int L, const float* d_uncond,
                                int Lu, double scale, int H, int W, float* d_pred, float* d_u, float* d_c, cudaStream_t caller);
void model_forward_diffuser_host(Ctx& c, const float* latent, int t, const float* context, int n, int L, const float* uncond,
                                 int Lu, double scale, int H, int W, float* pred, float* out_u, float* out_c);
void model_clip_forward_dev(Ctx& c, const int* d_tokens, int n, int L, float* d_out, cudaStream_t caller);
void model_clip_forward_host(Ctx& c, const int* tokens, int n, int L, float* out);
// dump-dir reader (dumpdir.cu)
bool npy_read_f32(const std::string& file, std::vector<float>& out);
long long dump_tensor_read(const std::string& file, int ndim, int64_t* dims, std::vector<float>& payload);
void model_load_dump_dir(Ctx& c, const char* root);
void model_test_attention(Ctx& c, const float* q, const float* k, const float* v, int n, int Nq, int Nk, int C, int heads,
                          float* out);

}  // namespace sdb
