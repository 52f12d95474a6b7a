// api.cu — extern "C" boundary (include/sdb200.h). No exception crosses it.
#include "../../include/sdb200.h"

#include <dlfcn.h>

#include <cstdlib>
#include <cstring>
#include <mutex>

#include "attention.cuh"
#include "kernels.cuh"
#include "model.cuh"
#include "runtime.cuh"

using namespace sdb;

struct sdb_ctx {
  Ctx c;
};

static thread_local std::string g_err;

#define API_BEGIN(ctxp)                      \
  if (!(ctxp)) {                             \
    g_err = "null context";                  \
    return 1;                                \
  }                                          \
  Ctx& c = (ctxp)->c;                        \
  try {                                      \
    SDB_CUDA(cudaSetDevice(c.device));

#define API_END                              \
  }                                          \
  catch (const std::exception& e) {          \
    c.err = e.what();                        \
    g_err = c.err;                           \
    return 1;                                \
  }                                          \
  return 0;

// one teardown for sdb_destroy and for a failed sdb_create (a context holds ~35 GB of device memory)
static void ctx_teardown(sdb_ctx* h) {
  if (!h) return;
  cudaSetDevice(h->c.device);
  cudaDeviceSynchronize();
  model_destroy(h->c);
  h->c.io_destroy();
  h->c.master.destroy();
  h->c.packed.destroy();
  h->c.work.destroy();
  if (h->c.stream) cudaStreamDestroy(h->c.stream);
  h->c.stream = nullptr;
  delete h;
}

// ------------------------------------------------------------------------------ NCCL, resolved at run time
// The library has no link-time dependency on NCCL: libnccl.so.2 is dlopen'ed by the first multi-GPU call (inside a torch
// process this binds to the copy torch already loaded, same SONAME). Only the four entry points used are declared.
namespace {
struct NcclApi {
  typedef struct { char internal[128]; } UniqueId;
  int (*GetUniqueId)(UniqueId*) = nullptr;
  int (*CommInitRank)(void** comm, int nranks, UniqueId id, int rank) = nullptr;
  int (*Broadcast)(const void* send, void* recv, size_t count, int dtype, int root, void* comm, cudaStream_t st) = nullptr;
  int (*CommDestroy)(void* comm) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(h, "ncclCommInitRank");
    api.Broadcast = (decltype(api.Broadcast))dlsym(h, "ncclBroadcast");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(h, "ncclCommDestroy");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(h, "ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.Broadcast && api.CommDestroy;
  });
  return api;
}
void nccl_check(int rc, const char* what) {
  if (rc != 0) {
    NcclApi& a = nccl();
    throw Error(std::string(what) + " failed: " + (a.GetErrorString ? a.GetErrorString(rc) : "nccl error " + std::to_string(rc)));
  }
}
}  // namespace

extern "C" {

const char* sdb_version(void) { return "sdb200 0.2.0 sm_100a"; }

int sdb_create(int device, sdb_ctx** out) {
  if (!out) {
    g_err = "null out pointer";
    return 1;
  }
  *out = nullptr;
  sdb_ctx* h = nullptr;
  try {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
      throw Error(std::string("no CUDA device available (") + cudaGetErrorString(e) +
                  "); this library has no CPU fallback");
    if (device < 0 || device >= ndev) throw Error("device index out of range");
    SDB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    SDB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
      throw Error(std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                  "; kernels are built for sm_100a only");
    h = new sdb_ctx();
    h->c.device = device;
    h->c.debug_sync = getenv("SDB_DEBUG_SYNC") && atoi(getenv("SDB_DEBUG_SYNC")) != 0;
    if (getenv("SDB_CLUSTER")) h->c.opt_cluster = atoi(getenv("SDB_CLUSTER"));
    if (getenv("SDB_PDL")) g_pdl_enabled = atoi(getenv("SDB_PDL")) != 0, g_pdl_late = atoi(getenv("SDB_PDL")) == 2;
    if (getenv("SDB_PAIR_BN256")) h->c.opt_pair_bn256 = atoi(getenv("SDB_PAIR_BN256"));
    SDB_CUDA(cudaStreamCreateWithFlags(&h->c.stream, cudaStreamNonBlocking));
    model_create(h->c);
    *out = h;
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    ctx_teardown(h);  // arenas, stream, model, tickets: nothing of a half-built context may leak
    return 1;
  }
}

int sdb_destroy(sdb_ctx* ctx) {
  ctx_teardown(ctx);
  return 0;
}

const char* sdb_last_error(sdb_ctx* ctx) { return ctx ? ctx->c.err.c_str() : g_err.c_str(); }

// ------------------------------------------------------------------------------ weights
int sdb_tensor_count(sdb_ctx* ctx) { return ctx ? (int)ctx->c.tensors.size() : -1; }

int sdb_tensor_info(sdb_ctx* ctx, int index, const char** name, int64_t dims[4], int* ndim) {
  API_BEGIN(ctx)
  SDB_CHECK(index >= 0 && index < (int)c.tensors.size(), "tensor index");
  const TensorInfo& t = c.tensors[index];
  if (name) *name = t.name.c_str();
  if (dims)
    for (int i = 0; i < 4; ++i) dims[i] = t.dims[i];
  if (ndim) *ndim = t.ndim;
  API_END
}

int sdb_set_tensor(sdb_ctx* ctx, const char* name, const float* host, const int64_t* dims, int ndim) {
  API_BEGIN(ctx)
  SDB_CHECK(name && host && dims, "null argument");
  const TensorInfo& t = c.info(name);
  SDB_CHECK(ndim == t.ndim, std::string("rank mismatch for ") + name);
  for (int i = 0; i < ndim; ++i) SDB_CHECK(dims[i] == t.dims[i], std::string("shape mismatch for ") + name);
  SDB_CUDA(cudaMemcpyAsync(c.master_ptr(name), host, t.count * sizeof(float), cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  c.finalized = false;
  API_END
}

int sdb_get_tensor(sdb_ctx* ctx, const char* name, float* host, int64_t count) {
  API_BEGIN(ctx)
  const TensorInfo& t = c.info(name);
  SDB_CHECK(count == t.count, "element count mismatch");
  SDB_CUDA(cudaMemcpyAsync(host, c.master_ptr(name), t.count * sizeof(float), cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

int sdb_load_dump_dir(sdb_ctx* ctx, const char* path) {
  API_BEGIN(ctx)
  model_load_dump_dir(c, path);
  API_END
}

int64_t sdb_read_dump_tensor(const char* file, int ndim, int64_t* dims, float* data, int64_t capacity) {
  try {
    SDB_CHECK(file && dims && ndim >= 1 && ndim <= 4, "bad argument");
    std::vector<float> payload;
    int64_t d[4];
    const long long count = dump_tensor_read(file, ndim, d, payload);
    for (int i = 0; i < ndim; ++i) dims[i] = d[i];
    if (data) {
      SDB_CHECK(capacity >= count, "buffer too small");
      std::memcpy(data, payload.data() + ndim, (size_t)count * sizeof(float));
    }
    return count;
  } catch (const std::exception& e) {
    g_err = e.what();
    return -1;
  }
}

int sdb_init_synthetic(sdb_ctx* ctx, uint32_t seed) {
  API_BEGIN(ctx)
  c.norm_eps.clear();
  model_init_synthetic(c, seed);
  c.finalized = false;
  API_END
}

int sdb_weight_arena(sdb_ctx* ctx, void** dev_ptr, size_t* bytes) {
  API_BEGIN(ctx)
  if (dev_ptr) *dev_ptr = c.master.base;
  if (bytes) *bytes = c.master.off;
  API_END
}

int sdb_nccl_unique_id(void* id128) {
  try {
    SDB_CHECK(id128, "null argument");
    SDB_CHECK(nccl().ok, "libnccl.so.2 not found: multi-GPU weight broadcast unavailable");
    NcclApi::UniqueId id;
    nccl_check(nccl().GetUniqueId(&id), "ncclGetUniqueId");
    std::memcpy(id128, &id, sizeof(id));
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 1;
  }
}

int sdb_broadcast_weights(sdb_ctx* ctx, const void* id128, int rank, int world) {
  API_BEGIN(ctx)
  SDB_CHECK(id128 && world >= 1 && rank >= 0 && rank < world, "broadcast_weights arguments");
  if (world > 1) {
    SDB_CHECK(nccl().ok, "libnccl.so.2 not found: multi-GPU weight broadcast unavailable");
    NcclApi::UniqueId id;
    std::memcpy(&id, id128, sizeof(id));
    void* comm = nullptr;
    nccl_check(nccl().CommInitRank(&comm, world, id, rank), "ncclCommInitRank");
    try {
      // (1) the fp32 master arena: every tensor of the registry in one contiguous block (dtype 7 = ncclFloat32)
      nccl_check(nccl().Broadcast(c.master.base, c.master.base, c.master.off / sizeof(float), 7, 0, comm, c.stream), "ncclBroadcast(arena)");
      // (2) the per-norm eps table a dump-dir carries beside the tensors (host map on rank 0): one float per registry tensor
      // (0 = default), so ranks that did not read the directory normalise with the same eps
      const size_t nt = c.tensors.size();
      std::vector<float> eps(nt, 0.f);
      if (rank == 0)
        for (size_t i = 0; i < nt; ++i)
          if (c.tensors[i].kind == K_NORM_G) {
            const std::string& nm = c.tensors[i].name;
            auto it = c.norm_eps.find(nm.substr(0, nm.rfind('/')));
            if (it != c.norm_eps.end()) eps[i] = it->second;
          }
      float* d_eps = (float*)c.io(5, nt * sizeof(float));
      SDB_CUDA(cudaMemcpyAsync(d_eps, eps.data(), nt * sizeof(float), cudaMemcpyHostToDevice, c.stream));
      nccl_check(nccl().Broadcast(d_eps, d_eps, nt, 7, 0, comm, c.stream), "ncclBroadcast(eps)");
      SDB_CUDA(cudaMemcpyAsync(eps.data(), d_eps, nt * sizeof(float), cudaMemcpyDeviceToHost, c.stream));
      SDB_CUDA(cudaStreamSynchronize(c.stream));
      if (rank != 0) {
        c.norm_eps.clear();
        for (size_t i = 0; i < nt; ++i)
          if (eps[i] > 0.f) {
            const std::string& nm = c.tensors[i].name;
            c.norm_eps[nm.substr(0, nm.rfind('/'))] = eps[i];
          }
      }
    } catch (...) {
      nccl().CommDestroy(comm);
      throw;
    }
    nccl_check(nccl().CommDestroy(comm), "ncclCommDestroy");
  }
  c.finalized = false;
  API_END
}

int sdb_finalize_weights(sdb_ctx* ctx) {
  API_BEGIN(ctx)
  model_finalize(c);
  c.finalized = true;
  API_END
}

// ------------------------------------------------------------------------------ hot path
static void need_final(Ctx& c) { SDB_CHECK(c.finalized, "call sdb_finalize_weights first"); }

int sdb_unet_forward(sdb_ctx* ctx, const float* x, int32_t timestep, const float* context, int n, int H, int W, int L,
                     float* out) {
  API_BEGIN(ctx)
  need_final(c);
  model_unet_forward_host(c, x, timestep, context, n, H, W, L, out);
  API_END
}

int sdb_unet_forward_dev(sdb_ctx* ctx, const float* d_x, int32_t timestep, const float* d_context, int n, int H, int W,
                         int L, float* d_out, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_unet_forward_dev(c, d_x, timestep, d_context, n, H, W, L, d_out, (cudaStream_t)stream);
  API_END
}

int sdb_decode_latent(sdb_ctx* ctx, const float* latent, int n, int H, int W, float* img) {
  API_BEGIN(ctx)
  need_final(c);
  model_decode_host(c, latent, n, H, W, img);
  API_END
}

int sdb_decode_latent_dev(sdb_ctx* ctx, const float* d_latent, int n, int H, int W, float* d_img, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_decode_dev(c, d_latent, n, H, W, d_img, (cudaStream_t)stream);
  API_END
}

int sdb_sample_latent(sdb_ctx* ctx, const float* context, int n, int L, const float* uncond, int Lu,
                      double guidance_scale, int n_steps, const float* init_latent, uint64_t seed, int H, int W,
                      float* latent_out) {
  API_BEGIN(ctx)
  need_final(c);
  model_sample_host(c, context, n, L, uncond, Lu, guidance_scale, n_steps, init_latent, seed, H, W, latent_out, nullptr);
  API_END
}

int sdb_latent_to_image(sdb_ctx* ctx, const float* latent, int n, int H, int W, uint8_t* rgb) {
  API_BEGIN(ctx)
  need_final(c);
  model_latent_to_image_host(c, latent, n, H, W, rgb);
  API_END
}

int sdb_sample_image(sdb_ctx* ctx, const float* context, int n, int L, const float* uncond, int Lu, double guidance_scale,
                     int n_steps, const float* init_latent, uint64_t seed, int H, int W, uint8_t* rgb) {
  API_BEGIN(ctx)
  need_final(c);
  model_sample_host(c, context, n, L, uncond, Lu, guidance_scale, n_steps, init_latent, seed, H, W, nullptr, rgb);
  API_END
}

int sdb_sample_image_dev(sdb_ctx* ctx, const float* d_context, int n, int L, const float* d_uncond, int Lu,
                         double guidance_scale, int n_steps, const float* d_init_latent, int H, int W, uint8_t* d_rgb,
                         void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_sample_dev(c, d_context, n, L, d_uncond, Lu, guidance_scale, n_steps, d_init_latent, H, W, nullptr, d_rgb,
                   (cudaStream_t)stream);
  API_END
}

int sdb_forward_diffuser(sdb_ctx* ctx, const float* latent, int32_t timestep, const float* context, int n, int L,
                         const float* uncond, int Lu, double guidance_scale, int H, int W, float* pred, float* out_uncond,
                         float* out_cond) {
  API_BEGIN(ctx)
  need_final(c);
  SDB_CHECK(latent && context && uncond, "null argument");
  model_forward_diffuser_host(c, latent, timestep, context, n, L, uncond, Lu, guidance_scale, H, W, pred, out_uncond, out_cond);
  API_END
}

int sdb_forward_diffuser_dev(sdb_ctx* ctx, const float* d_latent, int32_t timestep, const float* d_context, int n, int L,
                             const float* d_uncond, int Lu, double guidance_scale, int H, int W, float* d_pred, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_forward_diffuser_dev(c, d_latent, timestep, d_context, n, L, d_uncond, Lu, guidance_scale, H, W, d_pred, nullptr, nullptr,
                             (cudaStream_t)stream);
  API_END
}

int sdb_encode_image(sdb_ctx* ctx, const float* img, int n, int H, int W, float* latent) {
  API_BEGIN(ctx)
  need_final(c);
  SDB_CHECK(img && latent, "null argument");
  model_encode_host(c, img, n, H, W, latent);
  API_END
}

int sdb_encode_image_dev(sdb_ctx* ctx, const float* d_img, int n, int H, int W, float* d_latent, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_encode_dev(c, d_img, n, H, W, d_latent, (cudaStream_t)stream);
  API_END
}

int sdb_img2img(sdb_ctx* ctx, const uint8_t* rgb, const uint8_t* mask, const float* context, int n, int L, const float* uncond,
                int Lu, double guidance_scale, int n_steps, double strength, const float* noise, uint64_t seed, int H, int W,
                float* latent_out, uint8_t* rgb_out) {
  API_BEGIN(ctx)
  need_final(c);
  SDB_CHECK(context && uncond, "null argument");
  model_img2img_host(c, rgb, mask, context, n, L, uncond, Lu, guidance_scale, n_steps, strength, noise, seed, H, W, latent_out,
                     rgb_out);
  API_END
}

int sdb_img2img_dev(sdb_ctx* ctx, const uint8_t* d_rgb, const uint8_t* d_mask, const float* d_context, int n, int L,
                    const float* d_uncond, int Lu, double guidance_scale, int n_steps, double strength, const float* d_noise,
                    uint64_t seed, int H, int W, float* d_latent_out, uint8_t* d_rgb_out, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_img2img_dev(c, d_rgb, d_mask, d_context, n, L, d_uncond, Lu, guidance_scale, n_steps, strength, d_noise, seed, H, W,
                    d_latent_out, d_rgb_out, (cudaStream_t)stream);
  API_END
}

static_assert(SDB_SAMPLER_DDIM == SAMPLER_DDIM && SDB_SAMPLER_DPMPP_2M == SAMPLER_DPMPP_2M, "sampler ids of sdb200.h");

int sdb_sample_ex(sdb_ctx* ctx, const float* context, int n, int L, const float* uncond, int Lu, double guidance_scale,
                  int n_steps, int sampler, double eta, const float* init_latent, const float* step_noise, uint64_t seed, int H,
                  int W, float* latent_out, uint8_t* rgb_out) {
  API_BEGIN(ctx)
  need_final(c);
  SDB_CHECK(context && uncond, "null argument");
  model_sample_ex_host(c, context, n, L, uncond, Lu, guidance_scale, n_steps, sampler, eta, init_latent, step_noise, seed, H, W,
                       latent_out, rgb_out);
  API_END
}

int sdb_sample_ex_dev(sdb_ctx* ctx, const float* d_context, int n, int L, const float* d_uncond, int Lu, double guidance_scale,
                      int n_steps, int sampler, double eta, const float* d_init_latent, const float* d_step_noise, uint64_t seed,
                      int H, int W, float* d_latent_out, uint8_t* d_rgb_out, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_sample_ex_dev(c, d_context, n, L, d_uncond, Lu, guidance_scale, n_steps, sampler, eta, d_init_latent, d_step_noise, seed,
                      H, W, d_latent_out, d_rgb_out, (cudaStream_t)stream);
  API_END
}

int sdb_randn(sdb_ctx* ctx, uint64_t seed, int64_t count, float* out) {
  API_BEGIN(ctx)
  model_randn_host(c, seed, count, out);
  API_END
}

int sdb_clip_forward(sdb_ctx* ctx, const int32_t* tokens, int n, int L, float* out) {
  API_BEGIN(ctx)
  need_final(c);
  SDB_CHECK(tokens && out, "null argument");
  model_clip_forward_host(c, tokens, n, L, out);
  API_END
}

int sdb_clip_forward_dev(sdb_ctx* ctx, const int32_t* d_tokens, int n, int L, float* d_out, void* stream) {
  API_BEGIN(ctx)
  need_final(c);
  model_clip_forward_dev(c, d_tokens, n, L, d_out, (cudaStream_t)stream);
  API_END
}

// ------------------------------------------------------------------------------ options / profiling
int sdb_set_option(sdb_ctx* ctx, const char* key, int value) {
  API_BEGIN(ctx)
  const std::string k = key ? key : "";
  if (k == "precision")
    c.opt_precision = value;
  else if (k == "graphs")
    c.opt_graphs = value;
  else if (k == "splitk")
    c.opt_splitk = value;
  else if (k == "cluster")
    c.opt_cluster = value;
  else if (k == "pair_bn256")
    c.opt_pair_bn256 = value;
  else if (k == "raw16")
    c.opt_raw16 = value;
  else if (k == "splitk_min_iters")
    c.opt_splitk_min_iters = value;
  else if (k == "splitk_chunk")
    c.opt_splitk_chunk = value < 1 ? 1 : value;
  else if (k == "attn_split")
    c.opt_attn_split = value;
  else if (k == "attn_regsplit")
    g_attn_regsplit = value;
  else if (k == "emb_hoist")
    c.opt_emb_hoist = value;
  else if (k == "prefetch_w")
    c.opt_prefetch_w = value;
  else if (k == "mlp_passes")
    c.opt_mlp_passes = value;
  else if (k == "gn_epilogue")
    c.opt_gn_epilogue = value;
  else if (k == "skip_merge")
    c.opt_skip_merge = value;
  else if (k == "gn_apply_ctas")
    g_gn_apply_ctas = value < 1 ? 1 : value;
  else if (k == "gn_min_pix")
    g_gn_min_pix = value < 1 ? 1 : value;
  else
    throw Error("unknown option: " + k);
  model_invalidate_graphs(c);
  API_END
}

int sdb_profile_enable(sdb_ctx* ctx, int on) {
  API_BEGIN(ctx)
  profile_collect(c);
  c.profiling = on != 0;
  API_END
}
int sdb_profile_reset(sdb_ctx* ctx) {
  API_BEGIN(ctx)
  profile_collect(c);
  c.launches = 0;
  for (int i = 0; i < KC_COUNT; ++i) c.cls_ms[i] = c.cls_flops[i] = c.cls_bytes[i] = c.cls_issued[i] = 0, c.cls_launches[i] = 0;
  API_END
}
int sdb_profile_class_count(sdb_ctx*) { return KC_COUNT; }
int sdb_profile_get(sdb_ctx* ctx, int cls, const char** name, int64_t* launches, double* ms, double* flops, double* bytes) {
  API_BEGIN(ctx)
  SDB_CHECK(cls >= 0 && cls < KC_COUNT, "class index");
  profile_collect(c);
  if (name) *name = kernel_class_name(cls);
  if (launches) *launches = c.cls_launches[cls];
  if (ms) *ms = c.cls_ms[cls];
  if (flops) *flops = c.cls_flops[cls];
  if (bytes) *bytes = c.cls_bytes[cls];
  API_END
}
int sdb_profile_get_issued(sdb_ctx* ctx, int cls, double* issued_flops) {
  API_BEGIN(ctx)
  SDB_CHECK(cls >= 0 && cls < KC_COUNT && issued_flops, "class index");
  *issued_flops = c.cls_issued[cls];
  API_END
}
int64_t sdb_launch_count(sdb_ctx* ctx) { return ctx ? ctx->c.launches : -1; }

// ------------------------------------------------------------------------------ single-kernel test entries
// (host pointers; each call stages through the context's work arena)
int sdb_test_linear(sdb_ctx* ctx, const float* a, const float* w, const float* bias, int M, int K, int N, int passes,
                    float* out) {
  API_BEGIN(ctx)
  c.work.reset();
  float* d_a = c.work.get<float>((size_t)M * K);
  float* d_w = c.work.get<float>((size_t)K * N);
  float* d_b = bias ? c.work.get<float>(N) : nullptr;
  float* d_c = c.work.get<float>((size_t)M * N);
  SDB_CUDA(cudaMemcpyAsync(d_a, a, sizeof(float) * M * K, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_w, w, sizeof(float) * K * N, cudaMemcpyHostToDevice, c.stream));
  if (bias) SDB_CUDA(cudaMemcpyAsync(d_b, bias, sizeof(float) * N, cudaMemcpyHostToDevice, c.stream));
  ActOp A;
  A.p.hi = c.work.get<__half>((size_t)M * K);
  A.p.lo = c.work.get<__half>((size_t)M * K);
  A.W = M, A.C = K;
  WeightOp Wp;
  Wp.p.hi = c.work.get<__half>((size_t)N * K);
  Wp.p.lo = c.work.get<__half>((size_t)N * K);
  Wp.N = N, Wp.K = K;
  convert_f16_launch(d_a, (long long)M * K, A.p, c.stream);
  pack_linear_launch(d_w, K, N, Wp.p, 0, c.stream);
  Epilogue ep;
  ep.out_f32 = d_c;
  ep.bias = d_b;
  run_gemm(c, G_LINEAR, A, nullptr, Wp, passes, ep);
  SDB_CUDA(cudaMemcpyAsync(out, d_c, sizeof(float) * M * N, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

int sdb_test_gemm_ex(sdb_ctx* ctx, const float* a, const float* w, const float* bias, const float* residual, int M, int K, int N,
                     int passes, int flags, const float* xa, const float* xw, int XK, float* out) {
  API_BEGIN(ctx)
  c.work.reset();
  const bool geglu = flags & 1, from_f16 = flags & 4;
  SDB_CHECK(!geglu || (N % 128 == 0 && !residual && !xa), "GEGLU test: N (= 2 * hidden) must be a multiple of 128, no residual / extra K");
  const int Nout = geglu ? N / 2 : N;
  auto up = [&](const float* h, size_t cnt) {
    float* d = c.work.get<float>(cnt);
    SDB_CUDA(cudaMemcpyAsync(d, h, sizeof(float) * cnt, cudaMemcpyHostToDevice, c.stream));
    return d;
  };
  float* d_a = up(a, (size_t)M * K);
  float* d_w = up(w, (size_t)K * N);
  float* d_b = bias ? up(bias, N) : nullptr;
  float* d_r = residual ? up(residual, (size_t)M * N) : nullptr;
  float* d_c = c.work.get<float>((size_t)M * Nout);
  ActOp A;
  A.p = Half2Ptr{c.work.get<__half>((size_t)M * K), c.work.get<__half>((size_t)M * K)};
  A.W = M, A.C = K;
  convert_f16_launch(d_a, (long long)M * K, A.p, c.stream);
  WeightOp Wp;
  Wp.p = Half2Ptr{c.work.get<__half>((size_t)N * K), c.work.get<__half>((size_t)N * K)};
  Wp.N = N, Wp.K = K;
  float* d_bp = d_b;
  if (geglu) {
    SDB_CHECK(bias, "GEGLU test needs a bias");
    d_bp = c.work.get<float>(N);
    pack_geglu_launch(d_w, d_b, K, N / 2, 64, Wp.p, d_bp, c.stream);
  } else {
    pack_linear_launch(d_w, K, N, Wp.p, 0, c.stream);
  }
  ExtraK xk;
  if (xa) {
    SDB_CHECK(xw && XK % 64 == 0, "extra-K test operands");
    float* d_xa = up(xa, (size_t)M * XK);
    float* d_xw = up(xw, (size_t)XK * N);
    xk.x0.p = Half2Ptr{c.work.get<__half>((size_t)M * XK), c.work.get<__half>((size_t)M * XK)};
    xk.x0.W = M, xk.x0.C = XK;
    convert_f16_launch(d_xa, (long long)M * XK, xk.x0.p, c.stream);
    xk.w.p = Half2Ptr{c.work.get<__half>((size_t)N * XK), c.work.get<__half>((size_t)N * XK)};
    xk.w.N = N, xk.w.K = XK;
    pack_linear_launch(d_xw, XK, N, xk.w.p, 0, c.stream);
  }
  Epilogue ep;
  Half2Ptr o16;
  if (geglu || from_f16) o16 = Half2Ptr{c.work.get<__half>((size_t)M * Nout), c.work.get<__half>((size_t)M * Nout)};
  ep.out_f32 = geglu ? nullptr : d_c;
  ep.out_f16 = o16;
  ep.bias = d_bp, ep.residual = d_r, ep.geglu = geglu ? 1 : 0;
  run_gemm(c, G_LINEAR, A, nullptr, Wp, passes, ep, xa ? &xk : nullptr);
  if (geglu || from_f16) {
    std::vector<__half> hi((size_t)M * Nout), lo((size_t)M * Nout);
    SDB_CUDA(cudaMemcpyAsync(hi.data(), o16.hi, hi.size() * 2, cudaMemcpyDeviceToHost, c.stream));
    SDB_CUDA(cudaMemcpyAsync(lo.data(), o16.lo, lo.size() * 2, cudaMemcpyDeviceToHost, c.stream));
    SDB_CUDA(cudaStreamSynchronize(c.stream));
    for (size_t i = 0; i < hi.size(); ++i) out[i] = __half2float(hi[i]) + __half2float(lo[i]);
  } else {
    SDB_CUDA(cudaMemcpyAsync(out, d_c, sizeof(float) * M * Nout, cudaMemcpyDeviceToHost, c.stream));
    SDB_CUDA(cudaStreamSynchronize(c.stream));
  }
  API_END
}

int sdb_test_conv2d(sdb_ctx* ctx, const float* x, const float* w, const float* bias, int n, int cin, int H, int W,
                    int cout, int ksize, int stride, int upsample, int passes, float* y) {
  API_BEGIN(ctx)
  c.work.reset();
  SDB_CHECK(ksize == 1 || ksize == 3, "ksize");
  SDB_CHECK(stride == 1 || (stride == 2 && ksize == 3 && !upsample), "stride");
  const int Hin = H, Win = W;
  const int Ho = upsample ? 2 * H : (stride == 2 ? H / 2 : H), Wo = upsample ? 2 * W : (stride == 2 ? W / 2 : W);
  const size_t xin = (size_t)n * cin * Hin * Win, yout = (size_t)n * cout * Ho * Wo;
  float* d_x = c.work.get<float>(xin);
  float* d_xh = c.work.get<float>(xin);
  float* d_w = c.work.get<float>((size_t)cout * cin * ksize * ksize);
  float* d_b = bias ? c.work.get<float>(cout) : nullptr;
  float* d_yh = c.work.get<float>(yout);
  float* d_y = c.work.get<float>(yout);
  SDB_CUDA(cudaMemcpyAsync(d_x, x, sizeof(float) * xin, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_w, w, sizeof(float) * cout * cin * ksize * ksize, cudaMemcpyHostToDevice, c.stream));
  if (bias) SDB_CUDA(cudaMemcpyAsync(d_b, bias, sizeof(float) * cout, cudaMemcpyHostToDevice, c.stream));
  nchw_to_nhwc_launch(d_x, n, cin, Hin, Win, d_xh, c.stream);
  ActOp A;
  A.n = n, A.C = cin;
  WeightOp Wp;
  Wp.N = cout;
  int kind, mode = 0;
  if (ksize == 1) {
    kind = G_CONV1, A.H = Hin, A.W = Win;
    Wp.K = cin;
  } else if (stride == 2) {
    kind = G_CONV3_S2, mode = PREP_PHASE2, A.P = 4, A.H = Hin / 2, A.W = Win / 2;
    Wp.K = 9 * cin;
  } else if (upsample == 1) {
    kind = G_CONV3_UP2, A.H = Hin, A.W = Win;
    Wp.K = 4 * cin;
  } else if (upsample == 2) {
    kind = G_CONV3, mode = PREP_UP2, A.H = 2 * Hin, A.W = 2 * Win;
    Wp.K = 9 * cin;
  } else {
    kind = G_CONV3, A.H = Hin, A.W = Win;
    Wp.K = 9 * cin;
  }
  const size_t a_elems = (size_t)n * A.P * A.H * A.W * cin;
  A.p.hi = c.work.get<__half>(a_elems);
  A.p.lo = c.work.get<__half>(a_elems);
  const size_t w_elems = (size_t)cout * Wp.K * (kind == G_CONV3_UP2 ? 4 : 1);
  Wp.p.hi = c.work.get<__half>(w_elems);
  Wp.p.lo = c.work.get<__half>(w_elems);
  prep_operand_launch(d_xh, cin, nullptr, 0, n, Hin, Win, mode, nullptr, nullptr, nullptr, 0.f, A.p, c.stream);
  if (kind == G_CONV3_UP2)
    pack_conv_up2_launch(d_w, cout, cin, Wp.p, c.stream);
  else
    pack_conv_launch(d_w, cout, cin, ksize, Wp.p, c.stream);
  Epilogue ep;
  ep.out_f32 = d_yh;
  ep.bias = d_b;
  run_gemm(c, kind, A, nullptr, Wp, passes, ep);
  nhwc_to_nchw_launch(d_yh, n, cout, Ho, Wo, d_y, c.stream);
  SDB_CUDA(cudaMemcpyAsync(y, d_y, sizeof(float) * yout, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

int sdb_test_ln_fold(sdb_ctx* ctx, const float* a, const float* a2, const float* w0, const float* b0, const float* gamma,
                     const float* beta, const float* w1, const float* b1, int M, int K0, int C, int N, int passes, int geglu,
                     float* out) {
  API_BEGIN(ctx)
  c.work.reset();
  SDB_CHECK(C % 160 == 0 && K0 % 64 == 0 && (!geglu || (N % 128 == 0 && b1)), "ln_fold test shapes");
  auto up = [&](const float* h, size_t cnt) {
    float* d = c.work.get<float>(cnt);
    SDB_CUDA(cudaMemcpyAsync(d, h, sizeof(float) * cnt, cudaMemcpyHostToDevice, c.stream));
    return d;
  };
  auto h2 = [&](size_t cnt) { return Half2Ptr{c.work.get<__half>(cnt), c.work.get<__half>(cnt)}; };
  float *d_w0 = up(w0, (size_t)K0 * C), *d_b0 = up(b0, C), *d_g = up(gamma, C), *d_be = up(beta, C), *d_w1 = up(w1, (size_t)C * N);
  float* d_b1 = b1 ? up(b1, N) : nullptr;
  WeightOp W0;
  W0.p = h2((size_t)C * K0), W0.N = C, W0.K = K0;
  pack_linear_launch(d_w0, K0, C, W0.p, 0, c.stream);
  // consumer weights with gamma folded in, u / v vectors (the same recipe as pack_st)
  WeightOp W1;
  W1.p = h2((size_t)N * C), W1.N = N, W1.K = C;
  Half2Ptr scratch = h2((size_t)N * C);
  float *u_hi = c.work.get<float>(N), *u_full = c.work.get<float>(N), *v = c.work.get<float>(N), *bp = c.work.get<float>(N);
  if (geglu) {
    pack_geglu_launch(d_w1, d_b1, C, N / 2, 64, W1.p, bp, c.stream, d_g);
    pack_geglu_launch(d_w1, d_b1, C, N / 2, 64, scratch, nullptr, c.stream, d_be);
  } else {
    pack_linear_launch(d_w1, C, N, W1.p, 0, c.stream, 0, 0, d_g);
    pack_linear_launch(d_w1, C, N, scratch, 0, c.stream, 0, 0, d_be);
  }
  rowsum_f16_launch(W1.p, N, C, u_hi, u_full, c.stream);
  rowsum_f16_launch(scratch, N, C, nullptr, v, c.stream);
  if (geglu) add_vec_launch(v, bp, N, v, c.stream);
  else if (d_b1) add_vec_launch(v, d_b1, N, v, c.stream);
  // producer(s): y = a w0 + b0 (+ a2 w0 + b0 accumulated in place onto the fp16 pair), leaving row statistics
  Half2Ptr y16 = h2((size_t)M * C);
  const int ls = ln_slots(C);
  float* st = c.work.get<float>((size_t)M * ls * 2);
  for (int pass = 0; pass < (a2 ? 2 : 1); ++pass) {
    float* d_a = up(pass ? a2 : a, (size_t)M * K0);
    ActOp A;
    A.p = h2((size_t)M * K0), A.W = M, A.C = K0;
    convert_f16_launch(d_a, (long long)M * K0, A.p, c.stream);
    Epilogue ep;
    ep.out_f16 = y16, ep.bias = d_b0, ep.ln_out = st;
    if (pass) ep.residual16 = y16;
    run_gemm(c, G_LINEAR, A, nullptr, W0, 3, ep);
  }
  const int Nout = geglu ? N / 2 : N;
  Half2Ptr o16 = h2((size_t)M * Nout);
  {
    ActOp Y;
    Y.p = y16, Y.W = M, Y.C = C;
    Epilogue ep;
    ep.out_f16 = o16, ep.geglu = geglu ? 1 : 0;
    ep.ln_in = st, ep.ln_in_slots = ls, ep.ln_C = C, ep.ln_eps = 1e-5f, ep.ln_u_hi = u_hi, ep.ln_u_full = u_full, ep.bias = v;
    run_gemm(c, G_LINEAR, Y, nullptr, W1, passes, ep);
  }
  std::vector<__half> hi((size_t)M * Nout), lo((size_t)M * Nout);
  SDB_CUDA(cudaMemcpyAsync(hi.data(), o16.hi, hi.size() * 2, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaMemcpyAsync(lo.data(), o16.lo, lo.size() * 2, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  for (size_t i = 0; i < hi.size(); ++i) out[i] = __half2float(hi[i]) + __half2float(lo[i]);
  API_END
}

int sdb_test_conv_groupnorm(sdb_ctx* ctx, const float* x, const float* w, const float* bias, const float* gamma, const float* beta,
                            int n, int cin, int H, int W, int cout, int ksize, int passes, int silu, float* y, int* used_epilogue_stats) {
  API_BEGIN(ctx)
  c.work.reset();
  SDB_CHECK(ksize == 1 || ksize == 3, "ksize");
  const size_t xin = (size_t)n * cin * H * W, yout = (size_t)n * cout * H * W;
  auto up = [&](const float* h, size_t cnt) {
    float* d = c.work.get<float>(cnt);
    SDB_CUDA(cudaMemcpyAsync(d, h, sizeof(float) * cnt, cudaMemcpyHostToDevice, c.stream));
    return d;
  };
  float* d_x = up(x, xin);
  float* d_w = up(w, (size_t)cout * cin * ksize * ksize);
  float* d_b = bias ? up(bias, cout) : nullptr;
  float* d_g = up(gamma, cout);
  float* d_be = up(beta, cout);
  float* d_xh = c.work.get<float>(xin);
  float* d_conv = c.work.get<float>(yout);
  float* d_yh = c.work.get<float>(yout);
  float* d_y = c.work.get<float>(yout);
  nchw_to_nhwc_launch(d_x, n, cin, H, W, d_xh, c.stream);
  ActOp A;
  A.n = n, A.C = cin, A.H = H, A.W = W;
  A.p = Half2Ptr{c.work.get<__half>(xin), c.work.get<__half>(xin)};
  prep_operand_launch(d_xh, cin, nullptr, 0, n, H, W, 0, nullptr, nullptr, nullptr, 0.f, A.p, c.stream);
  WeightOp Wp;
  Wp.N = cout, Wp.K = ksize * ksize * cin;
  Wp.p = Half2Ptr{c.work.get<__half>((size_t)cout * Wp.K), c.work.get<__half>((size_t)cout * Wp.K)};
  pack_conv_launch(d_w, cout, cin, ksize, Wp.p, c.stream);
  GnPart gn;
  gn.bucket = cout % 320 == 0 ? 10 : cout / 32;
  gn.cap = std::max(3 * ((H * W + 127) / 128), 160);
  gn.buf = c.work.get<float>((size_t)n * gn.cap * (cout / gn.bucket) * 2);
  Epilogue ep;
  ep.out_f32 = d_conv, ep.bias = d_b, ep.gn = &gn;
  run_gemm(c, ksize == 1 ? G_CONV1 : G_CONV3, A, nullptr, Wp, passes, ep);
  if (used_epilogue_stats) *used_epilogue_stats = gn.slots;
  SDB_CHECK(gn.slots > 0, "the GEMM did not produce GroupNorm statistics for this shape");
  Half2Ptr o16{c.work.get<__half>(yout), c.work.get<__half>(yout)};
  GnSrc s0, s1;
  s0.x = d_conv, s0.C = cout, s0.part = gn.buf, s0.cap = gn.cap, s0.slots = gn.slots;
  gn_apply_launch(s0, s1, gn.bucket, n, H, W, silu, d_g, d_be, 1e-5f, o16, c.stream);
  std::vector<__half> hi(yout), lo(yout);
  SDB_CUDA(cudaMemcpyAsync(hi.data(), o16.hi, yout * 2, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaMemcpyAsync(lo.data(), o16.lo, yout * 2, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  std::vector<float> nhwc(yout);
  for (size_t i = 0; i < yout; ++i) nhwc[i] = __half2float(hi[i]) + __half2float(lo[i]);
  SDB_CUDA(cudaMemcpyAsync(d_yh, nhwc.data(), yout * 4, cudaMemcpyHostToDevice, c.stream));
  nhwc_to_nchw_launch(d_yh, n, cout, H, W, d_y, c.stream);
  SDB_CUDA(cudaMemcpyAsync(y, d_y, sizeof(float) * yout, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

int sdb_test_groupnorm(sdb_ctx* ctx, const float* x, const float* gamma, const float* beta, int n, int ch, int H, int W,
                       int silu, float* y) {
  API_BEGIN(ctx)
  c.work.reset();
  const size_t cnt = (size_t)n * ch * H * W;
  float* d_x = c.work.get<float>(cnt);
  float* d_xh = c.work.get<float>(cnt);
  float* d_yh = c.work.get<float>(cnt);
  float* d_y = c.work.get<float>(cnt);
  float* d_g = c.work.get<float>(ch);
  float* d_b = c.work.get<float>(ch);
  double* d_s = c.work.get<double>((size_t)n * 64);
  unsigned int* d_t = c.work.get<unsigned int>(n);
  float* d_p = c.work.get<float>(gn_stats_partial_floats(n, H * W));
  SDB_CUDA(cudaMemcpyAsync(d_x, x, sizeof(float) * cnt, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_g, gamma, sizeof(float) * ch, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_b, beta, sizeof(float) * ch, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemsetAsync(d_t, 0, sizeof(unsigned int) * n, c.stream));
  nchw_to_nhwc_launch(d_x, n, ch, H, W, d_xh, c.stream);
  gn_stats_launch(d_xh, ch, nullptr, 0, n, H * W, d_s, d_p, d_t, c.stream);
  gn_apply_f32_launch(d_xh, ch, n, H * W, silu, d_s, d_g, d_b, 1e-5f, d_yh, c.stream);
  nhwc_to_nchw_launch(d_yh, n, ch, H, W, d_y, c.stream);
  SDB_CUDA(cudaMemcpyAsync(y, d_y, sizeof(float) * cnt, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

int sdb_test_layernorm(sdb_ctx* ctx, const float* x, const float* gamma, const float* beta, int rows, int ch, float* y) {
  API_BEGIN(ctx)
  c.work.reset();
  const size_t cnt = (size_t)rows * ch;
  float* d_x = c.work.get<float>(cnt);
  float* d_y = c.work.get<float>(cnt);
  float* d_g = c.work.get<float>(ch);
  float* d_b = c.work.get<float>(ch);
  SDB_CUDA(cudaMemcpyAsync(d_x, x, sizeof(float) * cnt, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_g, gamma, sizeof(float) * ch, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_b, beta, sizeof(float) * ch, cudaMemcpyHostToDevice, c.stream));
  layernorm_launch(d_x, rows, ch, d_g, d_b, 1e-5f, Half2Ptr{}, d_y, c.stream);
  SDB_CUDA(cudaMemcpyAsync(y, d_y, sizeof(float) * cnt, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

int sdb_test_attention(sdb_ctx* ctx, const float* q, const float* k, const float* v, int n, int Nq, int Nk, int C,
                       int heads, float* out) {
  API_BEGIN(ctx)
  c.work.reset();
  model_test_attention(c, q, k, v, n, Nq, Nk, C, heads, out);
  API_END
}

}  // extern "C"
