// model.cu — the sampling graph: weight packing, UNet::forward, Autoencoder::decode_latent, DDIM sampler.
//
// Reference call stacks reproduced here (SURVEY §3):
//   StableDiffusion::sample_image / sample_latent / forward_diffuser  src/model/stablediffusion/mod.rs:51-192
//   UNet::forward                                                     src/model/unet/mod.rs:109-142
//   ResBlock / SpatialTransformer / TransformerBlock / MLP / MHA      src/model/unet/mod.rs:461-481,521-527,551-592,641-653,712-734
//   Autoencoder::decode_latent / Decoder / ResnetBlock / attention    src/model/autoencoder/mod.rs:68-71,204-217,307-324,513-528,562-608
// Activations are NHWC fp32 (residual stream); GEMM operands are staged as fp16 hi(/lo) tensors.
#include "model.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <functional>

#include "model_def.cuh"

namespace sdb {

static Model& M(Ctx& c) { return *reinterpret_cast<Model*>(c.model); }
static int round_up(int x, int m) { return (x + m - 1) / m * m; }

// tensor-core passes per product as a function of the UNet resolution level (0 = full latent resolution).
// Budgeted with the oracle's operand-rounding emulation (DESIGN.md "precision"): the two highest-resolution
// levels carry ~85 % of the fp16 rounding error of a UNet step, so they run the 3-term split product.
static int g_level_passes[4] = {3, 3, 1, 1};
// VAE decoder (same emulation study, per block): the latent-resolution stage (mid blocks, attention, first
// DecoderBlock) and the three upsample convs inject ~63 % of the fp16 rounding error for ~20 % of the FLOPs
// -> split product there, single pass on the 128^2..512^2 ResnetBlocks.
static int g_vae_passes_lowres = 3, g_vae_passes_up = 3, g_vae_passes_highres = 1;

// ================================================================================ packing
static Half2Ptr alloc_half2(Arena& a, size_t count) {
  Half2Ptr p;
  p.hi = a.get<__half>(count);
  p.lo = a.get<__half>(count);
  return p;
}
static float* mptr(Ctx& c, int idx) {
  return idx < 0 ? nullptr : reinterpret_cast<float*>(c.master.base) + c.tensors[idx].offset;
}

static void pack_conv(Ctx& c, ConvW& w, bool up2 = false) {
  w.bias = mptr(c, w.bi);
  if (w.cin % 64 != 0 || w.cout % 32 != 0) {  // CUDA-core convs
    if (w.cout <= 8 && w.k == 3 && w.cin % 4 == 0) {
      w.w_small = c.packed.get<float>((size_t)w.cout * 9 * w.cin);
      pack_small_cout_launch(mptr(c, w.wi), w.cout, w.cin, w.w_small, c.stream);
    }
    return;
  }
  if (up2) {
    w.packed.p = alloc_half2(c.packed, (size_t)16 * w.cout * w.cin);
    w.packed.N = w.cout, w.packed.K = 4 * w.cin;
    pack_conv_up2_launch(mptr(c, w.wi), w.cout, w.cin, w.packed.p, c.stream);
  } else {
    w.packed.p = alloc_half2(c.packed, (size_t)w.cout * w.k * w.k * w.cin);
    w.packed.N = w.cout, w.packed.K = w.k * w.k * w.cin;
    pack_conv_launch(mptr(c, w.wi), w.cout, w.cin, w.k, w.packed.p, c.stream);
  }
}
static void pack_lin(Ctx& c, LinW& w) {
  w.bias = mptr(c, w.bi);
  w.packed.p = alloc_half2(c.packed, (size_t)w.out * w.in);
  w.packed.N = w.out, w.packed.K = w.in;
  pack_linear_launch(mptr(c, w.wi), w.in, w.out, w.packed.p, 0, c.stream);
}
static void pack_norm(Ctx& c, NormW& n) {
  n.gamma = mptr(c, n.gi), n.beta = mptr(c, n.bi);
  const std::string& g = c.tensors[n.gi].name;
  auto it = c.norm_eps.find(g.substr(0, g.rfind('/')));
  n.eps = it == c.norm_eps.end() ? 1e-5f : it->second;
}

// [rows = heads*dpad][in]: head h occupies rows h*dpad .. h*dpad+d (pad rows stay zero)
static void pack_heads(Ctx& c, const LinW& src, int heads, int d, int dpad, Half2Ptr dst, int row_offset,
                       const float* in_scale = nullptr) {
  for (int h = 0; h < heads; ++h)
    pack_linear_launch(mptr(c, src.wi), src.in, d, dst, row_offset + h * dpad, c.stream, src.out, h * d, in_scale);
}

static void pack_resblock(Ctx& c, ResBlockW& r, int passes) {
  r.passes = passes;
  pack_norm(c, r.norm_in), pack_norm(c, r.norm_out);
  pack_conv(c, r.conv_in), pack_conv(c, r.conv_out);
  if (r.has_skip) {
    pack_conv(c, r.skip);
    r.bias_merged = c.packed.get<float>(r.cout);
    add_vec_launch(r.conv_out.bias, r.skip.bias, r.cout, r.bias_merged, c.stream);
  }
  r.lin_embed.bias = mptr(c, r.lin_embed.bi);
}
static void pack_st(Ctx& c, SpatialTransformerW& s, int passes) {
  s.passes = passes;
  pack_norm(c, s.norm), pack_norm(c, s.ln1), pack_norm(c, s.ln2), pack_norm(c, s.ln3);
  pack_conv(c, s.proj_in), pack_conv(c, s.proj_out);
  const int hd = s.heads * s.dpad;
  // The three LayerNorms of the TransformerBlock (unet/mod.rs:523-525) have no launch: gamma is folded into the weights of the
  // GEMM that consumes the normalised tensor (W' = diag(gamma) W), u = column sums of the packed W' (the exact fp16 values the
  // tensor cores multiply), v = beta^T W (+ bias); the GEMM reads the raw tensor and applies rstd * (acc - mean * u) + v.
  // The v vectors come from a scratch packing with beta in place of gamma (hi + lo = 22 bits of beta * W).
  Half2Ptr scratch = alloc_half2(c.work, (size_t)8 * s.c * s.c);
  auto fold = [&](WeightOp& w, float*& u_hi, float*& u_full, float*& v, const std::function<void(Half2Ptr, const float*)>& pack,
                  const NormW& ln) {
    pack(w.p, ln.gamma);
    u_hi = c.packed.get<float>(w.N), u_full = c.packed.get<float>(w.N), v = c.packed.get<float>(w.N);
    rowsum_f16_launch(w.p, w.N, w.K, u_hi, u_full, c.stream);
    SDB_CUDA(cudaMemsetAsync(scratch.hi, 0, (size_t)w.N * w.K * 2, c.stream));  // head-pad rows stay zero
    SDB_CUDA(cudaMemsetAsync(scratch.lo, 0, (size_t)w.N * w.K * 2, c.stream));
    pack(scratch, ln.beta);
    rowsum_f16_launch(scratch, w.N, w.K, nullptr, v, c.stream);
  };
  s.w_qkv1.p = alloc_half2(c.packed, (size_t)3 * hd * s.c), s.w_qkv1.N = 3 * hd, s.w_qkv1.K = s.c;
  fold(s.w_qkv1, s.u_qkv_hi, s.u_qkv_full, s.v_qkv, [&](Half2Ptr dst, const float* sc) {
    pack_heads(c, s.attn1.query, s.heads, s.d, s.dpad, dst, 0, sc);
    pack_heads(c, s.attn1.key, s.heads, s.d, s.dpad, dst, hd, sc);
    pack_heads(c, s.attn1.value, s.heads, s.d, s.dpad, dst, 2 * hd, sc);
  }, s.ln1);
  pack_lin(c, s.attn1.out), s.w_o1 = s.attn1.out.packed;
  s.w_q2.p = alloc_half2(c.packed, (size_t)hd * s.c), s.w_q2.N = hd, s.w_q2.K = s.c;
  fold(s.w_q2, s.u_q2_hi, s.u_q2_full, s.v_q2,
       [&](Half2Ptr dst, const float* sc) { pack_heads(c, s.attn2.query, s.heads, s.d, s.dpad, dst, 0, sc); }, s.ln2);
  s.w_kv2.p = alloc_half2(c.packed, (size_t)2 * hd * 768), s.w_kv2.N = 2 * hd, s.w_kv2.K = 768;
  pack_heads(c, s.attn2.key, s.heads, s.d, s.dpad, s.w_kv2.p, 0);
  pack_heads(c, s.attn2.value, s.heads, s.d, s.dpad, s.w_kv2.p, hd);
  pack_lin(c, s.attn2.out), s.w_o2 = s.attn2.out.packed;
  s.w_geglu.p = alloc_half2(c.packed, (size_t)8 * s.c * s.c), s.w_geglu.N = 8 * s.c, s.w_geglu.K = s.c;
  s.geglu_bias = c.packed.get<float>((size_t)8 * s.c);
  fold(s.w_geglu, s.u_geglu_hi, s.u_geglu_full, s.v_geglu, [&](Half2Ptr dst, const float* sc) {
    pack_geglu_launch(mptr(c, s.geglu.wi), mptr(c, s.geglu.bi), s.c, 4 * s.c, 64, dst, dst.hi == s.w_geglu.p.hi ? s.geglu_bias : nullptr,
                      c.stream, sc);
  }, s.ln3);
  add_vec_launch(s.v_geglu, s.geglu_bias, 8 * s.c, s.v_geglu, c.stream);  // v = beta^T W + b (packed order)
  pack_lin(c, s.ff);
  SDB_CUDA(cudaStreamSynchronize(c.stream));  // the scratch packing lives in the work arena
  c.work.reset();
}
static void pack_resnet(Ctx& c, ResnetW& r, int passes) {
  r.passes = passes;
  pack_norm(c, r.norm1), pack_norm(c, r.norm2);
  pack_conv(c, r.conv1), pack_conv(c, r.conv2);
  if (r.has_nin) {
    pack_conv(c, r.nin);
    r.bias_merged = c.packed.get<float>(r.cout);
    add_vec_launch(r.conv2.bias, r.nin.bias, r.cout, r.bias_merged, c.stream);
  }
}

void model_finalize(Ctx& c) {
  Model& m = M(c);
  model_invalidate_graphs(c);
  c.packed.reset();
  SDB_CUDA(cudaMemsetAsync(c.packed.base, 0, c.packed.cap, c.stream));  // head-pad rows must be zero
  // ---- UNet
  m.lin1_time.bias = mptr(c, m.lin1_time.bi), m.lin2_time.bias = mptr(c, m.lin2_time.bi);
  auto pack_block = [&](UNetBlockW& b) {
    const int p = g_level_passes[std::min(b.level, 3)];
    switch (b.kind) {
      case BK_CONV:
        pack_conv(c, b.conv);
        break;
      case BK_DOWN:
        pack_conv(c, b.conv), b.conv.passes = p;
        break;
      case BK_R:
        pack_resblock(c, b.res, p);
        break;
      case BK_RT:
        pack_resblock(c, b.res, p), pack_st(c, b.st, p);
        break;
      case BK_RU:
      case BK_RTU:
        pack_resblock(c, b.res, p);
        if (b.kind == BK_RTU) pack_st(c, b.st, p);
        pack_conv(c, b.conv, /*up2=*/true);
        b.conv.passes = g_level_passes[std::max(b.level - 1, 0)];  // the conv runs at the upsampled resolution
        break;
    }
  };
  for (auto& b : m.in_blocks) pack_block(b);
  pack_resblock(c, m.mid_res1, g_level_passes[3]);
  pack_st(c, m.mid_st, g_level_passes[3]);
  pack_resblock(c, m.mid_res2, g_level_passes[3]);
  for (auto& b : m.out_blocks) pack_block(b);
  pack_norm(c, m.norm_out);
  pack_conv(c, m.conv_out);
  // fused time-embedding projection: every lin_embed side by side, bias = lin bias + conv_in bias
  m.emb_total = 0;
  for (ResBlockW* r : m.resblocks) r->emb_off = m.emb_total, m.emb_total += r->cout;
  m.emb_w_all = c.packed.get<float>((size_t)1280 * m.emb_total);
  m.emb_b_all = c.packed.get<float>(m.emb_total);
  std::vector<float> hb(m.emb_total), t1, t2;
  for (ResBlockW* r : m.resblocks) {
    SDB_CUDA(cudaMemcpy2DAsync(m.emb_w_all + r->emb_off, (size_t)m.emb_total * 4, mptr(c, r->lin_embed.wi),
                               (size_t)r->cout * 4, (size_t)r->cout * 4, 1280, cudaMemcpyDeviceToDevice, c.stream));
    t1.resize(r->cout), t2.resize(r->cout);
    SDB_CUDA(cudaMemcpyAsync(t1.data(), mptr(c, r->lin_embed.bi), r->cout * 4, cudaMemcpyDeviceToHost, c.stream));
    SDB_CUDA(cudaMemcpyAsync(t2.data(), mptr(c, r->conv_in.bi), r->cout * 4, cudaMemcpyDeviceToHost, c.stream));
    SDB_CUDA(cudaStreamSynchronize(c.stream));
    for (int i = 0; i < r->cout; ++i) hb[r->emb_off + i] = t1[i] + t2[i];
  }
  SDB_CUDA(cudaMemcpyAsync(m.emb_b_all, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice, c.stream));
  // ---- VAE decoder
  pack_conv(c, m.post_quant), pack_conv(c, m.vae_conv_in), pack_conv(c, m.vae_conv_out);
  pack_resnet(c, m.mid_block1, g_vae_passes_lowres), pack_resnet(c, m.mid_block2, g_vae_passes_lowres);
  pack_norm(c, m.mid_attn.norm);
  pack_conv(c, m.mid_attn.q), pack_conv(c, m.mid_attn.k), pack_conv(c, m.mid_attn.v), pack_conv(c, m.mid_attn.proj_out);
  m.mid_attn.passes = g_vae_passes_lowres;
  for (int i = 0; i < 4; ++i) {
    for (int j = 0; j < 3; ++j) pack_resnet(c, m.dec[i].res[j], i == 0 ? g_vae_passes_lowres : g_vae_passes_highres);
    if (m.dec[i].has_up) pack_conv(c, m.dec[i].up, /*up2=*/true), m.dec[i].up.passes = g_vae_passes_up;
  }
  pack_norm(c, m.vae_norm_out);
  // ---- VAE encoder (row f4): every GEMM 3-term split-fp16 (runs once per image; no accuracy budget spent here)
  {
    EncoderW& e = m.enc;
    pack_conv(c, e.conv_in), pack_conv(c, e.conv_out), pack_conv(c, e.quant);
    // conv_in has 3 input channels: the Cin = 4 CUDA-core kernel gets weights padded with a zero fourth channel
    e.conv_in_w4 = c.packed.get<float>((size_t)128 * 36);
    SDB_CUDA(cudaMemsetAsync(e.conv_in_w4, 0, (size_t)128 * 36 * 4, c.stream));
    SDB_CUDA(cudaMemcpy2DAsync(e.conv_in_w4, 36 * 4, mptr(c, e.conv_in.wi), 27 * 4, 27 * 4, 128, cudaMemcpyDeviceToDevice, c.stream));
    for (int i = 0; i < 4; ++i) {
      pack_resnet(c, e.blocks[i].res[0], 3), pack_resnet(c, e.blocks[i].res[1], 3);
      if (e.blocks[i].has_down) pack_conv(c, e.blocks[i].down), e.blocks[i].down.passes = 3;
    }
    pack_resnet(c, e.mid_block1, 3), pack_resnet(c, e.mid_block2, 3);
    pack_norm(c, e.mid_attn.norm);
    pack_conv(c, e.mid_attn.q), pack_conv(c, e.mid_attn.k), pack_conv(c, e.mid_attn.v), pack_conv(c, e.mid_attn.proj_out);
    e.mid_attn.passes = 3;
    pack_norm(c, e.norm_out);
  }
  // ---- CLIP text encoder
  for (ClipBlockW& cb : m.clip.blocks) {
    pack_norm(c, cb.attn_ln), pack_norm(c, cb.mlp_ln);
    cb.w_qk.p = alloc_half2(c.packed, (size_t)2 * 768 * 768), cb.w_qk.N = 1536, cb.w_qk.K = 768;
    pack_linear_launch(mptr(c, cb.query.wi), 768, 768, cb.w_qk.p, 0, c.stream);
    pack_linear_launch(mptr(c, cb.key.wi), 768, 768, cb.w_qk.p, 768, c.stream);
    cb.bias_qk = c.packed.get<float>(1536);
    SDB_CUDA(cudaMemcpyAsync(cb.bias_qk, mptr(c, cb.query.bi), 768 * 4, cudaMemcpyDeviceToDevice, c.stream));
    SDB_CUDA(cudaMemcpyAsync(cb.bias_qk + 768, mptr(c, cb.key.bi), 768 * 4, cudaMemcpyDeviceToDevice, c.stream));
    pack_lin(c, cb.value), pack_lin(c, cb.out), pack_lin(c, cb.fc1), pack_lin(c, cb.fc2);
    // softmax rows sum to one, so P.(V + 1 b_v^T) = P.V + b_v^T: fold the value bias into the out-projection bias
    cb.bias_out = c.packed.get<float>(768);
    gemv_launch(mptr(c, cb.value.bi), mptr(c, cb.out.wi), mptr(c, cb.out.bi), 768, 768, cb.bias_out, c.stream);
  }
  pack_norm(c, m.clip.ln_final);
  // ---- schedule
  m.alphas_host.resize(1000);
  SDB_CUDA(cudaMemcpyAsync(m.alphas_host.data(), mptr(c, m.alphas_i), 4000, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  // a context filled through sdb_set_tensor without the schedule tensor would divide by sqrt(0) in every DDIM step
  for (float a : m.alphas_host)
    SDB_CHECK(a > 0.f && a <= 1.f, "alpha_cumulative_products must lie in (0, 1]: set the schedule tensor before sdb_finalize_weights");
}

void model_invalidate_graphs(Ctx& c) {
  Model& m = M(c);
  for (auto& g : m.graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  m.graphs.clear();
}

// ================================================================================ forward helpers
struct Act {
  float* p = nullptr;
  Half2Ptr raw16;  // optional fp16 hi/lo copy of the same values, written by the producing epilogue for consumers that
                   // read this tensor as a raw GEMM operand (skip 1x1 convs, upsample convs): no staging launch
  int n = 0, H = 0, W = 0, C = 0;
  GnPart gn;       // GroupNorm statistics left by the producing GEMM (gn.slots > 0 once a producer filled them)
  size_t count() const { return (size_t)n * H * W * C; }
};
// channel bucket of the producer-side GroupNorm statistics: must divide the group size of every GroupNorm that reads the tensor,
// alone or concatenated: 10 for the UNet widths (320/640/960/1280/1920/2560 -> groups of 10..80), C/32 for the VAE (128/256/512)
static int gn_bucket_of(int C) { return C % 320 == 0 ? 10 : (C % 32 == 0 ? C / 32 : 0); }

struct Fwd {
  Ctx& c;
  Model& m;
  int nb;
  double* gn_sums = nullptr;  // [slots][nb][32][2]
  unsigned int* gn_tickets = nullptr;  // [slots][nb]
  int gn_slot = 0, gn_slots = 0;
  Fwd(Ctx& c_, int nb_) : c(c_), m(M(c_)), nb(nb_) {}
  void init_sums(int slots) {
    gn_slots = slots;
    gn_sums = c.work.get<double>((size_t)slots * nb * 64);
    gn_tickets = c.work.get<unsigned int>((size_t)slots * nb * 2);  // one ticket counter per (slot, image); the second half is spare
    SDB_CUDA(cudaMemsetAsync(gn_tickets, 0, sizeof(unsigned int) * slots * nb * 2, c.stream));
  }
  // GroupNorm statistics of one tensor as [nb][32][2] sums (for the fused GroupNorm + SiLU + small-Cout convs): from the
  // producer's partials when it left any, else by reading the tensor
  double* stats(const Act& x) {
    SDB_CHECK(gn_slot < gn_slots, "GroupNorm statistics slots exhausted");
    double* sums = gn_sums + (size_t)gn_slot * nb * 64;
    unsigned int* tk = gn_tickets + (size_t)gn_slot * nb * 2;
    gn_slot++;
    const int HW = x.H * x.W;
    if (x.gn.slots > 0) {
      const int nbk = x.C / x.gn.bucket;
      const float* part = x.gn.buf;
      int cap = x.gn.cap, slots = x.gn.slots;
      if (slots > 128) {
        const int s2 = gn_fold_slots(slots);
        float* folded = c.work.get<float>((size_t)nb * s2 * nbk * 2);
        KernelScope ks(c, KC_GN_STATS, 0, (double)nb * slots * nbk * 8.0);
        gn_fold_launch(part, cap, slots, nbk, nb, folded, c.stream);
        part = folded, cap = s2, slots = s2;
      }
      KernelScope ks(c, KC_GN_STATS, 0, (double)nb * slots * nbk * 8.0);
      gn_sums_from_partials_launch(part, cap, slots, nbk, x.C, x.gn.bucket, nb, sums, c.stream);
      return sums;
    }
    float* part = c.work.get<float>(gn_stats_partial_floats(nb, HW));
    KernelScope ks(c, KC_GN_STATS, 0, (double)nb * HW * x.C * 4.0);
    gn_stats_launch(x.p, x.C, nullptr, 0, nb, HW, sums, part, tk, c.stream);
    return sums;
  }
  Act act16(int H, int W, int C) {
    Act a = act(H, W, C);
    if (c.opt_raw16) a.raw16 = half2(a.count(), true);
    return a;
  }
  ActOp raw16_operand(const Act& x) {
    ActOp a;
    a.n = nb, a.H = x.H, a.W = x.W, a.C = x.C, a.p = x.raw16;
    return a;
  }
  Act act(int H, int W, int C) {
    Act a;
    a.n = nb, a.H = H, a.W = W, a.C = C;
    a.p = c.work.get<float>(a.count());
    a.gn.bucket = gn_bucket_of(C);
    if (a.gn.bucket && c.opt_gn_epilogue) {
      a.gn.cap = std::max(3 * ((H * W + 127) / 128), 160);
      a.gn.buf = c.work.get<float>((size_t)nb * a.gn.cap * (C / a.gn.bucket) * 2);
    }
    return a;
  }
  Half2Ptr half2(size_t count, bool lo) {
    Half2Ptr p;
    p.hi = c.work.get<__half>(count);
    if (lo) p.lo = c.work.get<__half>(count);
    return p;
  }
  // GroupNorm(+SiLU) of cat(x0,x1) staged as an fp16 operand
  ActOp gn_operand(const Act& x0, const Act* x1, const NormW& nw, bool silu, bool lo) {
    const int C = x0.C + (x1 ? x1->C : 0);
    ActOp a;
    a.n = nb, a.H = x0.H, a.W = x0.W, a.C = C;
    a.p = half2((size_t)nb * x0.H * x0.W * C, lo);
    const int HW = x0.H * x0.W;
    if (x0.gn.slots > 0 && (!x1 || (x1->gn.slots > 0 && x1->gn.bucket == x0.gn.bucket)) && (C / 32) % x0.gn.bucket == 0) {
      GnSrc s0, s1;
      auto src = [&](const Act& x, GnSrc& s) {
        s.x = x.p, s.C = x.C, s.part = x.gn.buf, s.cap = x.gn.cap, s.slots = x.gn.slots;
        if (x.gn.slots > 128) {  // large image: shorten the per-CTA fold with a first pass over groups of 64 slots
          const int nbk = x.C / x.gn.bucket, s2 = gn_fold_slots(x.gn.slots);
          float* folded = c.work.get<float>((size_t)nb * s2 * nbk * 2);
          KernelScope ks(c, KC_GN_STATS, 0, (double)nb * x.gn.slots * nbk * 8.0);
          gn_fold_launch(x.gn.buf, x.gn.cap, x.gn.slots, nbk, nb, folded, c.stream);
          s.part = folded, s.cap = s2, s.slots = s2;
        }
      };
      src(x0, s0);
      if (x1) src(*x1, s1);
      KernelScope ks(c, KC_PREP, 0, (double)nb * HW * C * (4.0 + 2.0 + (lo ? 2.0 : 0.0)));
      gn_apply_launch(s0, s1, x0.gn.bucket, nb, x0.H, x0.W, silu ? 1 : 0, nw.gamma, nw.beta, nw.eps, a.p, c.stream);
      return a;
    }
    SDB_CHECK(gn_slot < gn_slots, "GroupNorm statistics slots exhausted");
    unsigned int* tk = gn_tickets + (size_t)gn_slot * nb * 2;
    gn_slot++;
    float* part = c.work.get<float>(gn_fused_partial_floats(nb, HW));
    KernelScope ks(c, KC_PREP, 0, (double)nb * HW * C * (8.0 + 2.0 + (lo ? 2.0 : 0.0)));
    gn_fused_launch(x0.p, x0.C, x1 ? x1->p : nullptr, x1 ? x1->C : 0, nb, x0.H, x0.W, silu ? 1 : 0, nw.gamma, nw.beta, nw.eps,
                    a.p, part, tk, c.stream);
    return a;
  }
  // raw (un-normalised) fp16 staging; mode 0, PREP_PHASE2 (stride-2 conv input)
  ActOp raw_operand(const Act& x0, const Act* x1, int mode, bool lo) {
    const int C = x0.C + (x1 ? x1->C : 0);
    ActOp a;
    a.n = nb, a.C = C;
    if (mode & PREP_PHASE2)
      a.P = 4, a.H = x0.H / 2, a.W = x0.W / 2;
    else
      a.H = x0.H, a.W = x0.W;
    a.p = half2((size_t)nb * x0.H * x0.W * C, lo);
    KernelScope ks(c, KC_PREP, 0, (double)x0.n * x0.H * x0.W * C * (4.0 + 2.0 + (lo ? 2.0 : 0.0)));
    prep_operand_launch(x0.p, x0.C, x1 ? x1->p : nullptr, x1 ? x1->C : 0, nb, x0.H, x0.W, mode, nullptr, nullptr, nullptr,
                        0.f, a.p, c.stream);
    return a;
  }
  ActOp rows_operand(Half2Ptr p, long long rows, int C) {
    ActOp a;
    a.p = p, a.n = 1, a.H = 1, a.W = (int)rows, a.C = C;
    return a;
  }
};

// reference unet/mod.rs:712-734 (emb_bias = conv_in.bias + lin_embed(silu(emb)); nullptr for the VAE ResnetBlock)
static void run_resblock(Fwd& f, const NormW& n1, const ConvW& c1, const NormW& n2, const ConvW& c2, const ConvW* skip,
                         const float* bias_merged, int passes, const Act& x0, const Act* x1, const float* emb_bias, Act& out) {
  Ctx& c = f.c;
  const size_t mark = c.work.off;
  const bool lo = passes >= 2 || c.opt_precision >= 2;
  ActOp a = f.gn_operand(x0, x1, n1, true, lo);
  ActOp raw, raw1;
  const bool have16 = x0.raw16.hi && (!lo || x0.raw16.lo) && (!x1 || (x1->raw16.hi && (!lo || x1->raw16.lo)));
  if (skip) {
    if (have16) {
      raw = f.raw16_operand(x0);
      if (x1) raw1 = f.raw16_operand(*x1);
    } else {
      raw = f.raw_operand(x0, x1, 0, lo);
    }
  }
  Act h = f.act(x0.H, x0.W, c1.cout);
  {
    Epilogue ep;
    ep.out_f32 = h.p, ep.gn = &h.gn;
    ep.bias = emb_bias ? emb_bias : c1.bias;
    run_gemm(c, G_CONV3, a, nullptr, c1.packed, passes, ep);
  }
  ActOp b = f.gn_operand(h, nullptr, n2, true, lo);
  // the 1x1 skip conv rides in conv_out's K loop when its inputs already exist as fp16 operands
  const bool merge = skip && have16 && bias_merged && c.opt_skip_merge;
  if (skip && !merge) {
    Epilogue ep;
    ep.out_f32 = out.p;
    ep.bias = skip->bias;
    run_gemm(c, G_CONV1, raw, (have16 && x1) ? &raw1 : nullptr, skip->packed, passes, ep);
  }
  {
    Epilogue ep;
    ep.out_f32 = out.p, ep.out_f16 = out.raw16, ep.gn = &out.gn;
    ExtraK xk;
    if (merge) {
      xk.x0 = raw, xk.has_x1 = x1 != nullptr, xk.w = skip->packed;
      if (x1) xk.x1 = raw1;
      ep.bias = bias_merged;
    } else {
      ep.bias = c2.bias;
      ep.residual = skip ? out.p : x0.p;  // in-place accumulate onto the skip-conv result, or + x
    }
    run_gemm(c, G_CONV3, b, nullptr, c2.packed, passes, ep, merge ? &xk : nullptr);
  }
  c.work.off = mark;  // temporaries are dead once the block's kernels are queued (stream order)
}

// per-layer K / V^T of the context tokens (constant over the DDIM steps)
struct CtxKV {
  __half* kv = nullptr;     // [nb*Lpad][2*heads*dpad]: K | V of the context tokens, head-padded
  __half* kv_lo = nullptr;  // lo halves (the split QK^T of the 3-pass levels reads K as a hi + lo pair)
};
struct CtxState {
  Half2Ptr ctx16;  // [nb*Lpad][768]
  int Lpad = 0;
  int* kvlen = nullptr;  // device [nb]
  std::vector<CtxKV> kv; // one per SpatialTransformer in execution order
};

// reference unet/mod.rs:461-481 + 521-527 + 641-653 + 551-592
// The block's residual stream y lives as an fp16 hi + lo pair (22 significant bits; no fp32 copy): every GEMM that reads it as
// an operand takes the pair as it is, every GEMM that adds to it reads and rewrites the pair in place. The three LayerNorms have
// no launch (see pack_st): the producers of y leave row statistics, the consumers normalise in their epilogue.
static void run_spatial_transformer(Fwd& f, SpatialTransformerW& s, const CtxState& cs, const CtxKV& kv, const Act& x,
                                    Act& out) {
  Ctx& c = f.c;
  const size_t mark = c.work.off;
  const int P = s.passes;
  const bool lo = P >= 2 || c.opt_precision >= 2;
  const int HW = x.H * x.W;
  const long long Mt = (long long)f.nb * HW;
  const int C = s.c, hd = s.heads * s.dpad;
  const int ls = ln_slots(C);
  // GroupNorm (no activation) -> proj_in (1x1 conv == GEMM over tokens)
  ActOp a = f.gn_operand(x, nullptr, s.norm, false, lo);
  Half2Ptr y16 = f.half2((size_t)Mt * C, true);
  float* st1 = c.work.get<float>((size_t)Mt * ls * 2);
  float* st2 = c.work.get<float>((size_t)Mt * ls * 2);
  float* st3 = c.work.get<float>((size_t)Mt * ls * 2);
  {
    Epilogue ep;
    ep.out_f16 = y16, ep.bias = s.proj_in.bias, ep.ln_out = st1;
    run_gemm(c, G_CONV1, a, nullptr, s.proj_in.packed, P, ep);
  }
  Half2Ptr o16 = f.half2((size_t)Mt * C, lo);
  auto ln_consume = [&](Epilogue& ep, const float* stats, const NormW& nw, const float* u_hi, const float* u_full, const float* v) {
    ep.ln_in = stats, ep.ln_in_slots = ls, ep.ln_C = C, ep.ln_eps = nw.eps, ep.ln_u_hi = u_hi, ep.ln_u_full = u_full, ep.bias = v;
  };
  // ---- self attention: x += out(attn(q,k,v = LN1(x))); one GEMM for q | k | v (head-padded columns), the attention kernel
  // takes V as it is written here (MN-major operand)
  // on the 3-pass levels q and k also get their lo halves: the attention kernel forms the logits as a 3-term split product
  const bool qk_split = lo && c.opt_attn_split && attention_supports_qk3(s.dpad);
  __half* qkv = c.work.get<__half>((size_t)Mt * 3 * hd);
  __half* qkv_lo = qk_split ? c.work.get<__half>((size_t)Mt * 3 * hd) : nullptr;
  {
    Epilogue ep;
    ep.out_f16.hi = qkv, ep.out_f16.lo = qkv_lo;
    ln_consume(ep, st1, s.ln1, s.u_qkv_hi, s.u_qkv_full, s.v_qkv);
    run_gemm(c, G_LINEAR, f.rows_operand(y16, Mt, C), nullptr, s.w_qkv1, P, ep);
  }
  {
    AttnOp at;
    at.q = qkv, at.ldq = 3 * hd, at.q_col0 = 0, at.q_rows = HW;
    at.k = qkv, at.ldk = 3 * hd, at.k_col0 = hd, at.k_rows = HW;
    at.vT = qkv, at.ldv = 3 * hd, at.v_mn = 1, at.v_col0 = 2 * hd;
    at.q_lo = qkv_lo, at.k_lo = qkv_lo;
    at.nb = f.nb, at.heads = s.heads, at.d = s.d, at.dpad = s.dpad, at.Nq = HW, at.Nk = HW;
    at.out = o16, at.ldo = C;
    run_attention(c, at);
  }
  {
    Epilogue ep;
    ep.out_f16 = y16, ep.residual16 = y16, ep.bias = s.attn1.out.bias, ep.ln_out = st2;
    run_gemm(c, G_LINEAR, f.rows_operand(o16, Mt, C), nullptr, s.w_o1, P, ep);
  }
  // ---- cross attention: x += out(attn(q = LN2(x), k,v = context))
  __half* q2 = c.work.get<__half>((size_t)Mt * hd);
  __half* q2_lo = qk_split ? c.work.get<__half>((size_t)Mt * hd) : nullptr;
  {
    Epilogue ep;
    ep.out_f16.hi = q2, ep.out_f16.lo = q2_lo;
    ln_consume(ep, st2, s.ln2, s.u_q2_hi, s.u_q2_full, s.v_q2);
    run_gemm(c, G_LINEAR, f.rows_operand(y16, Mt, C), nullptr, s.w_q2, P, ep);
  }
  {
    AttnOp at;
    at.q = q2, at.ldq = hd, at.q_col0 = 0, at.q_rows = HW;
    at.k = kv.kv, at.ldk = 2 * hd, at.k_col0 = 0, at.k_rows = cs.Lpad;
    at.vT = kv.kv, at.ldv = 2 * hd, at.v_mn = 1, at.v_col0 = hd;
    at.q_lo = q2_lo, at.k_lo = kv.kv_lo;
    at.nb = f.nb, at.heads = s.heads, at.d = s.d, at.dpad = s.dpad, at.Nq = HW, at.Nk = cs.Lpad;
    at.kvlen = cs.kvlen;
    at.out = o16, at.ldo = C;
    run_attention(c, at);
  }
  {
    Epilogue ep;
    ep.out_f16 = y16, ep.residual16 = y16, ep.bias = s.attn2.out.bias, ep.ln_out = st3;
    run_gemm(c, G_LINEAR, f.rows_operand(o16, Mt, C), nullptr, s.w_o2, P, ep);
  }
  // ---- GEGLU MLP: x += lin(x_a * gelu(gate)), LN3 folded into the GEGLU projection
  const int Pm = c.opt_mlp_passes ? c.opt_mlp_passes : P;  // pass policy of the MLP pair (DESIGN.md "precision")
  Half2Ptr g16 = f.half2((size_t)Mt * 4 * C, Pm >= 2 || c.opt_precision >= 2);
  {
    Epilogue ep;
    ep.geglu = 1, ep.out_f16 = g16;
    ln_consume(ep, st3, s.ln3, s.u_geglu_hi, s.u_geglu_full, s.v_geglu);
    run_gemm(c, G_LINEAR, f.rows_operand(y16, Mt, C), nullptr, s.w_geglu, Pm, ep);
  }
  {
    Epilogue ep;
    ep.out_f16 = y16, ep.residual16 = y16, ep.bias = s.ff.bias;
    run_gemm(c, G_LINEAR, f.rows_operand(g16, Mt, 4 * C), nullptr, s.ff.packed, Pm, ep);
  }
  // ---- proj_out + residual with the block input
  {
    Epilogue ep;
    ep.out_f32 = out.p, ep.out_f16 = out.raw16, ep.residual = x.p, ep.bias = s.proj_out.bias, ep.gn = &out.gn, ep.gn_rpi = HW;
    run_gemm(c, G_LINEAR, f.rows_operand(y16, Mt, C), nullptr, s.proj_out.packed, P, ep);
  }
  c.work.off = mark;
}

// context tokens -> fp16 + per-layer K / V^T (reference unet/mod.rs:646-647 with context = Some(..))
static void prepare_context(Fwd& f, const float* d_ctx /*[nb][Lpad][768] zero padded*/, int Lpad, int* d_kvlen,
                            CtxState& cs) {
  Ctx& c = f.c;
  Model& m = f.m;
  cs.Lpad = Lpad;
  cs.kvlen = d_kvlen;
  const long long rows = (long long)f.nb * Lpad;
  cs.ctx16 = f.half2((size_t)rows * 768, true);
  {
    KernelScope ks(c, KC_ELEMENTWISE);
    convert_f16_launch(d_ctx, rows * 768, cs.ctx16, c.stream);
  }
  cs.kv.resize(m.sts.size());
  for (size_t i = 0; i < m.sts.size(); ++i) {
    SpatialTransformerW& s = *m.sts[i];
    const int hd = s.heads * s.dpad;
    CtxKV& kv = cs.kv[i];
    kv.kv = c.work.get<__half>((size_t)rows * 2 * hd);
    kv.kv_lo = c.work.get<__half>((size_t)rows * 2 * hd);
    {
      Epilogue ep;
      ep.out_f16.hi = kv.kv, ep.out_f16.lo = kv.kv_lo;
      run_gemm(c, G_LINEAR, f.rows_operand(cs.ctx16, rows, 768), nullptr, s.w_kv2, 3, ep);
    }
  }
}

// ================================================================================ UNet::forward
struct UNetIO {
  const float* x;      // [nb,4,H,W] NCHW
  const int* t_dev;    // device scalar timestep
  float* out;          // [nb,4,H,W] NCHW
  int H, W;
  const float* emb_all = nullptr;  // [1000][emb_total] rows precomputed per timestep value (sample_latent), or null
};

static void unet_forward(Fwd& f, const UNetIO& io, const CtxState& cs) {
  Ctx& c = f.c;
  Model& m = f.m;
  const size_t mark0 = c.work.off;
  f.gn_slot = 0;
  f.init_sums(64);
  // ---- time embedding (unet/mod.rs:19-30, 115-118) and all 22 lin_embed rows in one GEMV (:718-722)
  float* emb_hidden = c.work.get<float>(1280);
  float* emb_silu = c.work.get<float>(1280);
  float* emb_rows = c.work.get<float>(m.emb_total);
  if (io.emb_all) {
    // the rows of this timestep were computed before the step loop (model_sample_dev): one copy instead of three GEMVs
    KernelScope ks(c, KC_ELEMENTWISE, 0.0, 8.0 * m.emb_total);
    emb_select_launch(io.emb_all, io.t_dev, m.emb_total, emb_rows, c.stream);
  } else {
    {
      KernelScope ks(c, KC_ELEMENTWISE);
      time_embed_launch(io.t_dev, mptr(c, m.lin1_time.wi), m.lin1_time.bias, mptr(c, m.lin2_time.wi), m.lin2_time.bias,
                        emb_hidden, emb_silu, c.stream);
    }
    {
      KernelScope ks(c, KC_ELEMENTWISE, 2.0 * 1280 * m.emb_total, 4.0 * 1280 * m.emb_total);
      gemv_launch(emb_silu, m.emb_w_all, m.emb_b_all, 1280, m.emb_total, emb_rows, c.stream);
    }
  }
  int st_index = 0;
  std::vector<Act> saved;
  Act x;
  int H = io.H, W = io.W;
  auto do_res = [&](ResBlockW& r, const Act& x0, const Act* x1, Act& o) {
    run_resblock(f, r.norm_in, r.conv_in, r.norm_out, r.conv_out, r.has_skip ? &r.skip : nullptr, r.bias_merged, r.passes, x0, x1,
                 emb_rows + r.emb_off, o);
  };
  auto do_block = [&](UNetBlockW& b, const Act& x0, const Act* x1) -> Act {
    Act o;
    switch (b.kind) {
      case BK_CONV: {
        o = f.act16(H, W, b.cout);
        KernelScope ks(c, KC_SMALLCONV, 2.0 * f.nb * H * W * 36.0 * b.cout);
        conv3x3_cin4_launch(io.x, f.nb, H, W, mptr(c, b.conv.wi), b.conv.bias, b.cout, nullptr, nullptr, 1.f, o.p, o.raw16,
                            c.stream);
        break;
      }
      case BK_DOWN: {  // unet/mod.rs:412-427: 3x3 stride 2 pad 1
        o = f.act16(H / 2, W / 2, b.cout);
        const size_t mk = c.work.off;
        const bool lo = b.conv.passes >= 2 || c.opt_precision >= 2;
        ActOp a = f.raw_operand(x0, nullptr, PREP_PHASE2, lo);
        Epilogue ep;
        ep.out_f32 = o.p, ep.out_f16 = o.raw16, ep.bias = b.conv.bias, ep.gn = &o.gn;
        run_gemm(c, G_CONV3_S2, a, nullptr, b.conv.packed, b.conv.passes, ep);
        c.work.off = mk;
        H /= 2, W /= 2;
        break;
      }
      case BK_R:
        o = f.act16(H, W, b.cout);
        do_res(b.res, x0, x1, o);
        break;
      case BK_RT: {
        o = f.act16(H, W, b.cout);
        Act r = f.act(H, W, b.cout);
        do_res(b.res, x0, x1, r);
        run_spatial_transformer(f, b.st, cs, cs.kv[st_index++], r, o);
        break;
      }
      case BK_RU:
      case BK_RTU: {
        o = f.act16(2 * H, 2 * W, b.cout);
        const size_t mk = c.work.off;
        // the tensor the upsample conv reads (resblock or transformer output) gets its fp16 copy from its producer
        Act r = b.kind == BK_RTU ? f.act(H, W, b.cout) : f.act16(H, W, b.cout);
        do_res(b.res, x0, x1, r);
        Act u = r;
        if (b.kind == BK_RTU) {
          u = f.act16(H, W, b.cout);
          run_spatial_transformer(f, b.st, cs, cs.kv[st_index++], r, u);
        }
        // unet/mod.rs:390-398: nearest 2x + conv3x3, folded into four 2x2-tap phase convolutions
        const bool lo = b.conv.passes >= 2 || c.opt_precision >= 2;
        ActOp a = u.raw16.hi ? f.raw16_operand(u) : f.raw_operand(u, nullptr, 0, lo);
        Epilogue ep;
        ep.out_f32 = o.p, ep.out_f16 = o.raw16, ep.bias = b.conv.bias, ep.gn = &o.gn;
        run_gemm(c, G_CONV3_UP2, a, nullptr, b.conv.packed, b.conv.passes, ep);
        // `o` was allocated before mk, so releasing the temporaries keeps it alive
        c.work.off = mk;
        H *= 2, W *= 2;
        break;
      }
    }
    return o;
  };
  // input blocks (unet/mod.rs:124-127)
  for (auto& b : m.in_blocks) {
    x = do_block(b, x, nullptr);
    saved.push_back(x);
  }
  // middle block (:130)
  {
    Act r1 = f.act(H, W, 1280), t = f.act(H, W, 1280), r2 = f.act16(H, W, 1280);
    do_res(m.mid_res1, x, nullptr, r1);
    run_spatial_transformer(f, m.mid_st, cs, cs.kv[st_index++], r1, t);
    do_res(m.mid_res2, t, nullptr, r2);
    x = r2;
  }
  // output blocks: x = cat([x, saved.pop()], 1) (:133-136) — the concat is never materialised in fp32
  for (auto& b : m.out_blocks) {
    Act skip = saved.back();
    saved.pop_back();
    x = do_block(b, x, &skip);
  }
  // out: GroupNorm + SiLU + conv 320 -> 4 (:138-140), fused, fp32 on CUDA cores, NCHW result
  {
    double* sums = f.stats(x);
    KernelScope ks(c, KC_SMALLCONV, 2.0 * f.nb * H * W * 9.0 * 320 * 4);
    conv3x3_small_cout_launch(x.p, f.nb, H, W, 320, sums, m.norm_out.gamma, m.norm_out.beta, m.norm_out.eps, m.conv_out.w_small,
                              m.conv_out.bias, 4, io.out, c.stream);
  }
  c.work.off = mark0;
}

// ================================================================================ VAE decoder
static void run_resnet(Fwd& f, ResnetW& r, const Act& x, Act& out) {
  run_resblock(f, r.norm1, r.conv1, r.norm2, r.conv2, r.has_nin ? &r.nin : nullptr, r.bias_merged, r.passes, x, nullptr, nullptr,
               out);
}

// reference autoencoder/mod.rs:562-608: 1 head, d = C = 512, N = H*W tokens. S is materialised per image
// (64 MB at 64x64) because the op runs once per image; q/k/v/proj are the same tcgen05 GEMMs.
static void run_vae_attention(Fwd& f, VaeAttnW& a, const Act& x, Act& out) {
  Ctx& c = f.c;
  const size_t mark = c.work.off;
  const int P = a.passes;
  const bool lo = P >= 2 || c.opt_precision >= 2;
  const int HW = x.H * x.W, C = x.C;
  const long long Mt = (long long)f.nb * HW;
  ActOp h = f.gn_operand(x, nullptr, a.norm, false, lo);
  const int Mp = round_up((int)Mt, 32);
  Half2Ptr q16 = f.half2((size_t)Mt * C, lo), k16 = f.half2((size_t)Mt * C, lo), vT = f.half2((size_t)C * Mp, lo);
  Half2Ptr o16 = f.half2((size_t)Mt * C, lo);
  {
    Epilogue ep;
    ep.out_f16 = q16, ep.bias = a.q.bias;
    run_gemm(c, G_CONV1, h, nullptr, a.q.packed, P, ep);
  }
  {
    Epilogue ep;
    ep.out_f16 = k16, ep.bias = a.k.bias;
    run_gemm(c, G_CONV1, h, nullptr, a.k.packed, P, ep);
  }
  {
    // V^T = Wv . h^T ; the v bias is added after P.V (softmax rows sum to one)
    WeightOp tok;
    tok.p = h.p, tok.N = Mp, tok.rows = (int)Mt, tok.K = C;
    Epilogue ep;
    ep.out_f16 = vT;
    run_gemm(c, G_LINEAR, f.rows_operand(a.v.packed.p, C, C), nullptr, tok, P, ep);
  }
  float* S = c.work.get<float>((size_t)HW * HW);
  Half2Ptr p16 = f.half2((size_t)HW * HW, lo);
  const float scale = (float)(1.0 / std::sqrt((double)C));
  for (int s = 0; s < f.nb; ++s) {
    Half2Ptr qs{q16.hi + (size_t)s * HW * C, q16.lo ? q16.lo + (size_t)s * HW * C : nullptr};
    WeightOp ks_;
    ks_.p.hi = k16.hi + (size_t)s * HW * C, ks_.p.lo = k16.lo ? k16.lo + (size_t)s * HW * C : nullptr;
    ks_.N = HW, ks_.K = C;
    {
      Epilogue ep;
      ep.out_f32 = S;
      run_gemm(c, G_LINEAR, f.rows_operand(qs, HW, C), nullptr, ks_, P, ep);
    }
    {
      KernelScope ks(c, KC_ELEMENTWISE, 0, (double)HW * HW * 6.0);
      softmax_rows_launch(S, HW, HW, scale, p16, c.stream);
    }
    WeightOp vs;
    vs.p.hi = vT.hi + (size_t)s * HW, vs.p.lo = vT.lo ? vT.lo + (size_t)s * HW : nullptr;
    vs.N = C, vs.K = HW, vs.ld = Mp;
    Epilogue ep;
    ep.out_f16.hi = o16.hi + (size_t)s * HW * C, ep.out_f16.lo = o16.lo ? o16.lo + (size_t)s * HW * C : nullptr;
    ep.bias = a.v.bias;
    run_gemm(c, G_LINEAR, f.rows_operand(p16, HW, HW), nullptr, vs, P, ep);
  }
  {
    Epilogue ep;
    ep.out_f32 = out.p, ep.residual = x.p, ep.bias = a.proj_out.bias, ep.gn = &out.gn, ep.gn_rpi = HW;
    run_gemm(c, G_LINEAR, f.rows_operand(o16, Mt, C), nullptr, a.proj_out.packed, P, ep);
  }
  c.work.off = mark;
}

// latent [nb,4,H,W] NCHW (already divided by 0.18215 when called from latent_to_image) -> img [nb,3,8H,8W] NCHW
static void vae_decode(Fwd& f, const float* d_latent, int H, int W, float pre_scale, float* d_img) {
  Ctx& c = f.c;
  Model& m = f.m;
  const size_t mark0 = c.work.off;
  f.gn_slot = 0;
  f.init_sums(40);
  // post_quant_conv (1x1, 4->4) folded into conv_in's input gather (autoencoder/mod.rs:68-71, 205)
  Act x = f.act(H, W, 512);
  {
    KernelScope ks(c, KC_SMALLCONV, 2.0 * f.nb * H * W * 36.0 * 512);
    conv3x3_cin4_launch(d_latent, f.nb, H, W, mptr(c, m.vae_conv_in.wi), m.vae_conv_in.bias, 512, mptr(c, m.post_quant.wi),
                        m.post_quant.bias, pre_scale, x.p, Half2Ptr{}, c.stream);
  }
  // Mid (autoencoder/mod.rs:456-463)
  {
    Act a = f.act(H, W, 512), b = f.act(H, W, 512), d = f.act(H, W, 512);
    run_resnet(f, m.mid_block1, x, a);
    run_vae_attention(f, m.mid_attn, a, b);
    run_resnet(f, m.mid_block2, b, d);
    x = d;
  }
  // DecoderBlocks (autoencoder/mod.rs:307-324)
  for (int i = 0; i < 4; ++i) {
    DecoderBlockW& db = m.dec[i];
    for (int j = 0; j < 3; ++j) {
      // the tensor the upsampler reads gets its fp16 hi/lo copy from the producing epilogue
      Act o = (j == 2 && db.has_up) ? f.act16(H, W, db.res[j].cout) : f.act(H, W, db.res[j].cout);
      run_resnet(f, db.res[j], x, o);
      x = o;
    }
    if (db.has_up) {
      Act o = f.act16(2 * H, 2 * W, db.up.cout);  // read raw by the next block's nin_shortcut
      const size_t mk = c.work.off;
      const bool lo = db.up.passes >= 2 || c.opt_precision >= 2;
      ActOp a = x.raw16.hi ? f.raw16_operand(x) : f.raw_operand(x, nullptr, 0, lo);
      Epilogue ep;
      ep.out_f32 = o.p, ep.out_f16 = o.raw16, ep.bias = db.up.bias, ep.gn = &o.gn;
      run_gemm(c, G_CONV3_UP2, a, nullptr, db.up.packed, db.up.passes, ep);
      c.work.off = mk;
      x = o;
      H *= 2, W *= 2;
    }
  }
  // norm_out + SiLU + conv_out 128 -> 3 (autoencoder/mod.rs:215-216)
  {
    double* sums = f.stats(x);
    KernelScope ks(c, KC_SMALLCONV, 2.0 * f.nb * H * W * 9.0 * 128 * 3);
    conv3x3_small_cout_launch(x.p, f.nb, H, W, 128, sums, m.vae_norm_out.gamma, m.vae_norm_out.beta, m.vae_norm_out.eps,
                              m.vae_conv_out.w_small, m.vae_conv_out.bias, 3, d_img, c.stream);
  }
  c.work.off = mark0;
}

// ================================================================================ VAE encoder (SURVEY §8f row f4)
// Autoencoder::encode_image (autoencoder/mod.rs:60-66): Encoder::forward (:133-145) -> quant_conv -> channels [0,4).
// d_img4: the image with a zero fourth plane [nb][4][H][W]; d_latent [nb][4][H/8][W/8].
static void vae_encode(Fwd& f, const float* d_img4, int H, int W, float* d_latent) {
  Ctx& c = f.c;
  EncoderW& e = f.m.enc;
  const size_t mark0 = c.work.off;
  f.gn_slot = 0;
  f.init_sums(40);
  Act x = f.act(H, W, 128);
  {
    KernelScope ks(c, KC_SMALLCONV, 2.0 * f.nb * H * W * 27.0 * 128);
    conv3x3_cin4_launch(d_img4, f.nb, H, W, e.conv_in_w4, e.conv_in.bias, 128, nullptr, nullptr, 1.f, x.p, Half2Ptr{}, c.stream);
  }
  // EncoderBlocks (:255-265): two ResnetBlocks, then the stride-2 conv padded bottom/right only
  for (int i = 0; i < 4; ++i) {
    EncoderBlockW& eb = e.blocks[i];
    for (int j = 0; j < 2; ++j) {
      Act o = f.act(H, W, eb.res[j].cout);
      run_resnet(f, eb.res[j], x, o);
      x = o;
    }
    if (eb.has_down) {
      SDB_CHECK(H % 2 == 0 && W % 2 == 0, "encode_image: image height and width must be multiples of 8");
      Act o = f.act(H / 2, W / 2, eb.down.cout);
      const size_t mk = c.work.off;
      ActOp a = f.raw_operand(x, nullptr, PREP_PHASE2, true);
      Epilogue ep;
      ep.out_f32 = o.p, ep.bias = eb.down.bias, ep.gn = &o.gn;
      run_gemm(c, G_CONV3_S2_PAD01, a, nullptr, eb.down.packed, eb.down.passes, ep);
      c.work.off = mk;
      x = o;
      H /= 2, W /= 2;
    }
  }
  // Mid (:456-463)
  {
    Act a = f.act(H, W, 512), b = f.act(H, W, 512), d = f.act(H, W, 512);
    run_resnet(f, e.mid_block1, x, a);
    run_vae_attention(f, e.mid_attn, a, b);
    run_resnet(f, e.mid_block2, b, d);
    x = d;
  }
  // norm_out + SiLU + conv_out 512 -> 8 (fp32 CUDA cores, NCHW), then quant_conv 8 -> 8 and the slice [0,4)
  float* y8 = c.work.get<float>((size_t)f.nb * 8 * H * W);
  {
    double* sums = f.stats(x);
    KernelScope ks(c, KC_SMALLCONV, 2.0 * f.nb * H * W * 9.0 * 512 * 8);
    conv3x3_small_cout_launch(x.p, f.nb, H, W, 512, sums, e.norm_out.gamma, e.norm_out.beta, e.norm_out.eps, e.conv_out.w_small,
                              e.conv_out.bias, 8, y8, c.stream);
  }
  {
    KernelScope ks(c, KC_ELEMENTWISE);
    quant_conv_slice_launch(y8, mptr(c, e.quant.wi), e.quant.bias, f.nb, H * W, d_latent, c.stream);
  }
  c.work.off = mark0;
}

// ================================================================================ public entry points
namespace {
struct StreamJoin {  // run on c.stream ordered after / before the caller's stream
  Ctx& c;
  cudaStream_t caller;
  cudaEvent_t ev = nullptr;
  StreamJoin(Ctx& c_, cudaStream_t s) : c(c_), caller(s) {
    if (caller != c.stream) {
      SDB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      SDB_CUDA(cudaEventRecord(ev, caller));
      SDB_CUDA(cudaStreamWaitEvent(c.stream, ev, 0));
    }
  }
  ~StreamJoin() {
    if (ev) {
      cudaEventRecord(ev, c.stream);
      cudaStreamWaitEvent(caller, ev, 0);
      cudaEventDestroy(ev);
    }
  }
};
}  // namespace

// UNet pass over nb samples with per-sample context lengths. d_ctx_padded [nb][Lpad][768].
static void unet_pass(Ctx& c, int nb, const float* d_x, const int* d_t, const float* d_ctx_padded, int Lpad, int* d_kvlen,
                      int H, int W, float* d_out, const CtxState* shared_cs, const float* emb_all = nullptr) {
  Fwd f(c, nb);
  const size_t mark = c.work.off;
  CtxState local;
  const CtxState* cs = shared_cs;
  if (!cs) {
    prepare_context(f, d_ctx_padded, Lpad, d_kvlen, local);
    cs = &local;
  }
  UNetIO io{d_x, d_t, d_out, H, W};
  io.emb_all = emb_all;
  unet_forward(f, io, *cs);
  c.work.off = mark;
}

void model_unet_forward_dev(Ctx& c, const float* d_x, int t, const float* d_context, int n, int H, int W, int L,
                            float* d_out, cudaStream_t caller) {
  SDB_CHECK(n >= 1 && H % 8 == 0 && W % 8 == 0 && L >= 1, "unet_forward arguments");
  // the deepest level has (H/8)*(W/8) tokens per sample; TMA tile origins inside the V^T matrix are
  // per-sample column offsets and must stay 16-byte aligned
  SDB_CHECK(((H / 8) * (W / 8)) % 8 == 0, "unsupported latent size: (H/8)*(W/8) must be a multiple of 8");
  StreamJoin join(c, caller);
  c.work.reset();
  const int Lpad = round_up(L, 32);
  float* ctxp = c.work.get<float>((size_t)n * Lpad * 768);
  int* d_t = c.work.get<int>(1);
  int* d_len = c.work.get<int>(n);
  std::vector<int> lens(n, L);
  SDB_CUDA(cudaMemsetAsync(ctxp, 0, (size_t)n * Lpad * 768 * 4, c.stream));
  SDB_CUDA(cudaMemcpy2DAsync(ctxp, (size_t)Lpad * 768 * 4, d_context, (size_t)L * 768 * 4, (size_t)L * 768 * 4, n,
                             cudaMemcpyDeviceToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_t, &t, 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_len, lens.data(), 4 * n, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));  // host staging buffers (t, lens) must outlive the copies
  unet_pass(c, n, d_x, d_t, ctxp, Lpad, d_len, H, W, d_out, nullptr);
}

void model_unet_forward_host(Ctx& c, const float* x, int t, const float* context, int n, int H, int W, int L, float* out) {
  const size_t xe = (size_t)n * 4 * H * W, ce = (size_t)n * L * 768;
  float* d_x = (float*)c.io(0, xe * 4);
  float* d_c = (float*)c.io(1, ce * 4);
  float* d_o = (float*)c.io(2, xe * 4);
  SDB_CUDA(cudaMemcpyAsync(d_x, x, xe * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_c, context, ce * 4, cudaMemcpyHostToDevice, c.stream));
  model_unet_forward_dev(c, d_x, t, d_c, n, H, W, L, d_o, c.stream);
  SDB_CUDA(cudaMemcpyAsync(out, d_o, xe * 4, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

static void decode_chunked(Ctx& c, const float* d_latent, int n, int H, int W, float pre_scale, float* d_img) {
  // bounded working set: at most 4 images of 128-channel 8Hx8W activations at a time
  const int chunk = 4;
  for (int i = 0; i < n; i += chunk) {
    const int nb = std::min(chunk, n - i);
    Fwd f(c, nb);
    vae_decode(f, d_latent + (size_t)i * 4 * H * W, H, W, pre_scale, d_img + (size_t)i * 3 * 64 * H * W);
  }
}

void model_decode_dev(Ctx& c, const float* d_latent, int n, int H, int W, float* d_img, cudaStream_t caller) {
  StreamJoin join(c, caller);
  c.work.reset();
  decode_chunked(c, d_latent, n, H, W, 1.0f, d_img);
}

void model_decode_host(Ctx& c, const float* latent, int n, int H, int W, float* img) {
  const size_t le = (size_t)n * 4 * H * W, ie = (size_t)n * 3 * 64 * H * W;
  float* d_l = (float*)c.io(0, le * 4);
  float* d_i = (float*)c.io(1, ie * 4);
  SDB_CUDA(cudaMemcpyAsync(d_l, latent, le * 4, cudaMemcpyHostToDevice, c.stream));
  model_decode_dev(c, d_l, n, H, W, d_i, c.stream);
  SDB_CUDA(cudaMemcpyAsync(img, d_i, ie * 4, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

static void check_encode_size(int n, int H, int W) {
  SDB_CHECK(n >= 1 && H >= 64 && W >= 64 && H % 8 == 0 && W % 8 == 0 && ((H / 8) * (W / 8)) % 8 == 0,
            "encode_image: height and width must be multiples of 8, at least 64, with (H/8)*(W/8) a multiple of 8");
}

void model_encode_dev(Ctx& c, const float* d_img, int n, int H, int W, float* d_latent, cudaStream_t caller) {
  check_encode_size(n, H, W);
  StreamJoin join(c, caller);
  c.work.reset();
  const size_t plane = (size_t)H * W;
  for (int i0 = 0; i0 < n; i0 += 4) {  // chunks of 4 images bound the work arena like decode_chunked
    const int nb = std::min(4, n - i0);
    const size_t mark = c.work.off;
    float* img4 = c.work.get<float>((size_t)nb * 4 * plane);
    SDB_CUDA(cudaMemsetAsync(img4, 0, (size_t)nb * 4 * plane * 4, c.stream));
    SDB_CUDA(cudaMemcpy2DAsync(img4, 4 * plane * 4, d_img + (size_t)i0 * 3 * plane, 3 * plane * 4, 3 * plane * 4, nb,
                               cudaMemcpyDeviceToDevice, c.stream));
    Fwd f(c, nb);
    vae_encode(f, img4, H, W, d_latent + (size_t)i0 * 4 * (plane / 64));
    c.work.off = mark;
  }
}

void model_encode_host(Ctx& c, const float* img, int n, int H, int W, float* latent) {
  const size_t ie = (size_t)n * 3 * H * W, le = (size_t)n * 4 * (H / 8) * (W / 8);
  float* d_i = (float*)c.io(0, ie * 4);
  float* d_l = (float*)c.io(1, le * 4);
  SDB_CUDA(cudaMemcpyAsync(d_i, img, ie * 4, cudaMemcpyHostToDevice, c.stream));
  model_encode_dev(c, d_i, n, H, W, d_l, c.stream);
  SDB_CUDA(cudaMemcpyAsync(latent, d_l, le * 4, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

// latent_to_image (stablediffusion/mod.rs:69-100). With a pixel mask [n,8H,8W], pixels whose mask is 0 are copied from
// paste_rgb [n,8H,8W,3] instead (inpainting keeps the known image byte for byte).
static void latent_to_image_dev(Ctx& c, const float* d_latent, int n, int H, int W, uint8_t* d_rgb,
                                const uint8_t* paste_rgb = nullptr, const uint8_t* paste_mask = nullptr) {
  float* d_img = c.work.get<float>((size_t)n * 3 * 64 * H * W);
  // `latent * (1.0 / 0.18215)`: the scalar is rounded to f32 before the multiply, as burn's mul_scalar does
  decode_chunked(c, d_latent, n, H, W, (float)(1.0 / 0.18215), d_img);
  KernelScope ks(c, KC_ELEMENTWISE);
  if (paste_mask)
    to_rgb8_paste_launch(d_img, n, 8 * H, 8 * W, paste_rgb, paste_mask, d_rgb, c.stream);
  else
    to_rgb8_launch(d_img, n, 8 * H, 8 * W, d_rgb, c.stream);
}

void model_latent_to_image_host(Ctx& c, const float* latent, int n, int H, int W, uint8_t* rgb) {
  const size_t le = (size_t)n * 4 * H * W, re = (size_t)n * 3 * 64 * H * W;
  float* d_l = (float*)c.io(0, le * 4);
  uint8_t* d_r = (uint8_t*)c.io(1, re);
  c.work.reset();
  SDB_CUDA(cudaMemcpyAsync(d_l, latent, le * 4, cudaMemcpyHostToDevice, c.stream));
  latent_to_image_dev(c, d_l, n, H, W, d_r);
  SDB_CUDA(cudaMemcpyAsync(rgb, d_r, re, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

static void check_sample_args(int n, int L, int Lu, int n_steps, int H, int W) {
  SDB_CHECK(n >= 1 && L >= 1 && Lu >= 1, "sample arguments");
  SDB_CHECK(n_steps >= 1 && n_steps <= 1000, "n_steps must be in [1,1000] (step_by(0) panics in the reference)");
  SDB_CHECK(H % 8 == 0 && W % 8 == 0, "latent size must be a multiple of 8");
  SDB_CHECK(((H / 8) * (W / 8)) % 8 == 0, "unsupported latent size: (H/8)*(W/8) must be a multiple of 8");
}

// timesteps (stablediffusion/mod.rs:111,123): (0..1000).rev().step_by(1000 / n_steps)
static std::vector<int> ddim_timesteps(int n_steps) {
  std::vector<int> ts;
  for (int t = 999; t >= 0; t -= 1000 / n_steps) ts.push_back(t);
  return ts;
}

// Where a sampler run starts and what it blends (img2img / inpainting, DESIGN.md §7 row f5). The default is text-to-image.
struct SampleStart {
  int i0 = 0;                  // index of the first timestep of ddim_timesteps(n_steps) that runs
  const float* x0 = nullptr;   // [n,4,H,W] encoded image: the start latent is fl(fl(a*x0) + fl(b*eps)) at ts[i0]
  const float* eps = nullptr;  // [n,4,H,W] noise of the start latent and of the kept cells
  const uint8_t* m = nullptr;  // [n,H,W] latent mask (0 = keep the known image) or null: no blend
};

// The update each step applies (DESIGN.md §7 row f6; oracle/sampler_oracle.py states it). The default is the reference's
// DDIM at eta = 0, which keeps cfg_ddim_kernel and its arguments.
struct SamplerDesc {
  int kind = SAMPLER_DDIM;
  double eta = 0.0;                   // DDIM only
  const float* step_noise = nullptr;  // [T][n,4,H,W] z of DDIM with eta > 0, or null: the stream of sampler_step_seed(seed, i)
  uint64_t seed = 0;
  float* hist = nullptr;              // [n,4,H,W] x0 of the previous step (DPM-Solver++(2M))
};

uint64_t sampler_step_seed(uint64_t seed, int i) { return seed ^ ((uint64_t)(i + 1) * 0x9E3779B97F4A7C15ull); }

static double half_log_snr(double a) { return std::log(std::sqrt(a) / std::sqrt(1.0 - a)); }

// The DDIM / CFG loop of sample_latent over ts[st.i0:]. Leaves the final latent in the first half of the batch-2n input it
// returns, with the work arena at the mark after the step state, so the caller can decode from there. The work-arena layout
// depends on (n, L, Lu, H, W) only: every start index, blend state and sampler replays the same cached step graph.
static float* sample_loop(Ctx& c, const float* d_context, int n, int L, const float* d_uncond, int Lu, double scale,
                          int n_steps, const float* d_init_latent, const SampleStart& st, int H, int W,
                          const SamplerDesc& sd = SamplerDesc{}) {
  Model& m = M(c);
  c.work.reset();
  const int nb = 2 * n;
  const int Lpad = round_up(std::max(L, Lu), 32);
  const size_t le = (size_t)n * 4 * H * W;
  // batch layout: samples [0,n) = unconditional context, [n,2n) = prompt context
  float* ctxp = c.work.get<float>((size_t)nb * Lpad * 768);
  float* xb = c.work.get<float>(2 * le);
  float* eps = c.work.get<float>(2 * le);
  int* d_t = c.work.get<int>(1024);
  int* d_len = c.work.get<int>(nb);
  SDB_CUDA(cudaMemsetAsync(ctxp, 0, (size_t)nb * Lpad * 768 * 4, c.stream));
  for (int i = 0; i < n; ++i)
    SDB_CUDA(cudaMemcpyAsync(ctxp + (size_t)i * Lpad * 768, d_uncond, (size_t)Lu * 768 * 4, cudaMemcpyDeviceToDevice, c.stream));
  SDB_CUDA(cudaMemcpy2DAsync(ctxp + (size_t)n * Lpad * 768, (size_t)Lpad * 768 * 4, d_context, (size_t)L * 768 * 4,
                             (size_t)L * 768 * 4, n, cudaMemcpyDeviceToDevice, c.stream));
  const int step = 1000 / n_steps;
  std::vector<int> ts = ddim_timesteps(n_steps);
  SDB_CHECK(st.i0 >= 0 && st.i0 < (int)ts.size(), "sampler start index");
  ts.erase(ts.begin(), ts.begin() + st.i0);
  if (st.x0) {
    // x_t0 = sqrt(a[t0]) x0 + sqrt(1 - a[t0]) eps with the coefficients widened to f64 like the DDIM update's
    const double a0 = (double)m.alphas_host[ts[0]];
    KernelScope ks(c, KC_ELEMENTWISE);
    noise_latent_launch(st.x0, st.eps, (long long)le, (float)std::sqrt(a0), (float)std::sqrt(1.0 - a0), xb, c.stream);
  } else {
    SDB_CUDA(cudaMemcpyAsync(xb, d_init_latent, le * 4, cudaMemcpyDeviceToDevice, c.stream));
    SDB_CUDA(cudaMemcpyAsync(xb + le, d_init_latent, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  }
  std::vector<int> lens(nb);
  for (int i = 0; i < nb; ++i) lens[i] = i < n ? Lu : L;
  SDB_CUDA(cudaMemcpyAsync(d_t, ts.data(), ts.size() * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_len, lens.data(), nb * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));

  // time-embedding rows of every timestep of the schedule, once per call (unet/mod.rs:19-30, 115-118, 718-722 depend on t alone).
  // Fixed-size table indexed by the timestep value: the addresses of everything allocated after it do not depend on n_steps,
  // which the cached step graphs rely on.
  float* emb_all = nullptr;
  if (c.opt_emb_hoist) {
    emb_all = c.work.get<float>((size_t)1000 * m.emb_total);
    const size_t mk = c.work.off;
    float* hid = c.work.get<float>(ts.size() * 1280);
    float* sil = c.work.get<float>(ts.size() * 1280);
    {
      KernelScope ks(c, KC_ELEMENTWISE, 2.0 * 1280 * m.emb_total * ts.size(), 4.0 * 1280 * m.emb_total * ((ts.size() + 4) / 5));
      time_embed_rows_launch(d_t, (int)ts.size(), mptr(c, m.lin1_time.wi), m.lin1_time.bias, mptr(c, m.lin2_time.wi),
                             m.lin2_time.bias, m.emb_w_all, m.emb_b_all, m.emb_total, hid, sil, emb_all, c.stream);
    }
    c.launches += 2;  // three launches under one scope
    c.work.off = mk;  // stream order: the temporaries are dead before anything else is written there
  }

  Fwd f(c, nb);
  CtxState cs;
  prepare_context(f, ctxp, Lpad, d_len, cs);  // context K/V: once per image, not once per step

  // one CUDA graph of the UNet step per (nb,H,W,Lpad); replayed with a different timestep slot each step
  const long long key = ((long long)nb << 48) ^ ((long long)H << 36) ^ ((long long)W << 24) ^ ((long long)Lpad << 8) ^
                        (long long)(c.opt_precision & 3);
  const bool use_graph = c.opt_graphs && !c.profiling;
  int* d_tcur = c.work.get<int>(1);
  const size_t work_mark = c.work.off;
  cudaGraphExec_t exec = nullptr;
  int64_t graph_launches = 0;
  if (use_graph) {
    // the graph bakes in every work-arena address allocated after work_mark: a layout change must never replay it
    for (auto& g : m.graphs)
      if (g.key == key && g.io[0] == (void*)xb && g.io[1] == (void*)eps && g.io[2] == (void*)cs.kv[0].kv &&
          g.io[4] == (void*)(uintptr_t)work_mark)
        exec = g.exec, graph_launches = (int64_t)(intptr_t)g.io[3];
    if (!exec) {
      // warm-up pass outside capture (sets kernel attributes), then capture
      SDB_CUDA(cudaMemcpyAsync(d_tcur, d_t, 4, cudaMemcpyDeviceToDevice, c.stream));
      unet_pass(c, nb, xb, d_tcur, nullptr, Lpad, d_len, H, W, eps, &cs, emb_all);
      SDB_CUDA(cudaStreamSynchronize(c.stream));
      const int64_t before = c.launches;
      cudaGraph_t graph;
      SDB_CUDA(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
      try {
        unet_pass(c, nb, xb, d_tcur, nullptr, Lpad, d_len, H, W, eps, &cs, emb_all);
      } catch (...) {
        cudaGraph_t g2;
        cudaStreamEndCapture(c.stream, &g2);
        throw;
      }
      SDB_CUDA(cudaStreamEndCapture(c.stream, &graph));
      graph_launches = c.launches - before;
      c.launches = before;
      SDB_CUDA(cudaGraphInstantiate(&exec, graph, 0));
      cudaGraphDestroy(graph);
      Model::GraphEntry ge;
      ge.key = key, ge.exec = exec;
      memset(ge.io, 0, sizeof(ge.io));
      ge.io[0] = xb, ge.io[1] = eps, ge.io[2] = cs.kv[0].kv, ge.io[3] = (void*)(intptr_t)graph_launches;
      ge.io[4] = (void*)(uintptr_t)work_mark;
      m.graphs.push_back(ge);
    }
  }
  double h_prev = 0.0;  // DPM-Solver++(2M): h of the previous step
  for (size_t i = 0; i < ts.size(); ++i) {
    const int t = ts[i];
    // alphas are read as f32 and widened to f64 (stablediffusion/mod.rs:124-140)
    const double a_t = (double)m.alphas_host[t];
    const double a_prev = (t >= step) ? (double)m.alphas_host[t - step] : 1.0;
    SDB_CUDA(cudaMemcpyAsync(d_tcur, d_t + i, 4, cudaMemcpyDeviceToDevice, c.stream));
    if (exec) {
      SDB_CUDA(cudaGraphLaunch(exec, c.stream));
      c.launches += graph_launches;
    } else {
      c.work.off = work_mark;
      unet_pass(c, nb, xb, d_tcur, nullptr, Lpad, d_len, H, W, eps, &cs, emb_all);
    }
    KernelScope ks(c, KC_ELEMENTWISE);
    if (sd.kind == SAMPLER_DPMPP_2M) {
      // x0 = (x - pred*s_t)/alpha_t; h = lambda_next - lambda_t; x' = (s_next/s_t) x - alpha_next expm1(-h) D, D = x0 at
      // step 0, (1 + 1/2r) x0 - (1/2r) x0_prev with r = h_prev/h after it; the last step (a_next = 1) returns x0
      int kind = 2;
      double ratio = 0, coef = 0, w0 = 0, w1 = 0;
      if (a_prev < 1.0) {
        const double h = half_log_snr(a_prev) - half_log_snr(a_t);
        ratio = std::sqrt(1.0 - a_prev) / std::sqrt(1.0 - a_t), coef = std::sqrt(a_prev) * std::expm1(-h);
        kind = i == 0 ? 0 : 1;
        if (kind == 1) w0 = 1.0 + 1.0 / (2.0 * (h_prev / h)), w1 = 1.0 / (2.0 * (h_prev / h));
        h_prev = h;
      }
      cfg_dpmpp2m_launch(kind, eps, eps + le, xb, sd.hist, (long long)le, (float)scale, (float)std::sqrt(1.0 - a_t),
                         (float)std::sqrt(a_t), (float)ratio, (float)coef, (float)w0, (float)w1, c.stream);
    } else if (sd.eta > 0.0) {
      // sigma = eta sqrt((1 - a_next)/(1 - a_t)) sqrt(1 - a_t/a_next), 0 at the last step; x' = x0 sqrt(a_next) +
      // pred sqrt(1 - a_next - sigma^2) + sigma z (stablediffusion/mod.rs:152-155 with sigma != 0)
      const int si = st.i0 + (int)i;
      const double sigma = sd.eta * std::sqrt((1.0 - a_prev) / (1.0 - a_t)) * std::sqrt(1.0 - a_t / a_prev);
      cfg_ddim_eta_launch(eps, eps + le, xb, (long long)le, (float)scale, (float)std::sqrt(1.0 - a_t), (float)std::sqrt(a_t),
                          (float)std::sqrt(a_prev), (float)std::sqrt(std::max(0.0, 1.0 - a_prev - sigma * sigma)), (float)sigma,
                          sd.step_noise ? sd.step_noise + (size_t)si * le : nullptr, sampler_step_seed(sd.seed, si), c.stream);
    } else if (st.m)
      cfg_ddim_blend_launch(eps, eps + le, xb, (long long)le, (float)scale, (float)std::sqrt(1.0 - a_t), (float)std::sqrt(a_t),
                            (float)std::sqrt(a_prev), (float)std::sqrt(1.0 - a_prev), st.x0, st.eps, st.m, H * W, c.stream);
    else
      cfg_ddim_launch(eps, eps + le, xb, (long long)le, (float)scale, (float)std::sqrt(1.0 - a_t), (float)std::sqrt(a_t),
                      (float)std::sqrt(a_prev), (float)std::sqrt(1.0 - a_prev), c.stream);
  }
  c.work.off = work_mark;
  return xb;
}

// sample_latent + latent_to_image (stablediffusion/mod.rs:51-160). The conditional and unconditional UNet
// evaluations of a step (forward_diffuser :162-192) run as ONE batch-2n pass: weights stream from HBM once.
void model_sample_dev(Ctx& c, const float* d_context, int n, int L, const float* d_uncond, int Lu, double scale,
                      int n_steps, const float* d_init_latent, int H, int W, float* d_latent_out, uint8_t* d_rgb,
                      cudaStream_t caller) {
  check_sample_args(n, L, Lu, n_steps, H, W);
  StreamJoin join(c, caller);
  float* xb = sample_loop(c, d_context, n, L, d_uncond, Lu, scale, n_steps, d_init_latent, SampleStart{}, H, W);
  const size_t le = (size_t)n * 4 * H * W;
  if (d_latent_out) SDB_CUDA(cudaMemcpyAsync(d_latent_out, xb, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  if (d_rgb) latent_to_image_dev(c, xb, n, H, W, d_rgb);
}

// ---- selectable samplers (DESIGN.md §7 row f6): DDIM with eta in [0, 1] and DPM-Solver++(2M) on the reference's schedule.
// The reference fixes sigma = 0 (stablediffusion/mod.rs:119); oracle/sampler_oracle.py states both samplers once.
static void check_sample_ex_args(const void* latent_out, const void* rgb_out, int n, int L, int Lu, int n_steps, int sampler,
                                 double eta, const float* step_noise, int H, int W) {
  SDB_CHECK(sampler == SAMPLER_DDIM || sampler == SAMPLER_DPMPP_2M,
            "sample_ex: unknown sampler " + std::to_string(sampler) + " (0 = DDIM, 1 = DPM-Solver++(2M))");
  SDB_CHECK(eta >= 0.0 && eta <= 1.0, "sample_ex: eta must lie in [0, 1]");  // false for NaN
  SDB_CHECK(sampler == SAMPLER_DDIM || eta == 0.0, "sample_ex: eta applies to DDIM only (DPM-Solver++(2M) takes eta = 0)");
  SDB_CHECK(!step_noise || (sampler == SAMPLER_DDIM && eta > 0.0), "sample_ex: step_noise is used only by DDIM with eta > 0");
  SDB_CHECK(latent_out || rgb_out, "sample_ex: latent_out and rgb_out are both null");
  check_sample_args(n, L, Lu, n_steps, H, W);
}

void model_sample_ex_dev(Ctx& c, const float* d_context, int n, int L, const float* d_uncond, int Lu, double scale, int n_steps,
                         int sampler, double eta, const float* d_init_latent, const float* d_step_noise, uint64_t seed, int H, int W,
                         float* d_latent_out, uint8_t* d_rgb, cudaStream_t caller) {
  check_sample_ex_args(d_latent_out, d_rgb, n, L, Lu, n_steps, sampler, eta, d_step_noise, H, W);
  StreamJoin join(c, caller);
  const size_t le = (size_t)n * 4 * H * W;
  // the seeded initial latent and the DPM++ history live in Ctx::state: the work arena keeps the layout of every other sampler
  if (!d_init_latent) {
    float* l = (float*)c.state(4, le * 4);
    KernelScope ks(c, KC_ELEMENTWISE);
    randn_launch(l, (long long)le, seed, c.stream);  // the stream sdb_sample_latent draws its initial latent from
    d_init_latent = l;
  }
  SamplerDesc sd;
  sd.kind = sampler, sd.eta = eta, sd.step_noise = d_step_noise, sd.seed = seed;
  if (sampler == SAMPLER_DPMPP_2M) sd.hist = (float*)c.state(3, le * 4);
  float* xb = sample_loop(c, d_context, n, L, d_uncond, Lu, scale, n_steps, d_init_latent, SampleStart{}, H, W, sd);
  if (d_latent_out) SDB_CUDA(cudaMemcpyAsync(d_latent_out, xb, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  if (d_rgb) latent_to_image_dev(c, xb, n, H, W, d_rgb);
}

void model_sample_ex_host(Ctx& c, const float* context, int n, int L, const float* uncond, int Lu, double scale, int n_steps,
                          int sampler, double eta, const float* init_latent, const float* step_noise, uint64_t seed, int H, int W,
                          float* latent_out, uint8_t* rgb) {
  check_sample_ex_args(latent_out, rgb, n, L, Lu, n_steps, sampler, eta, step_noise, H, W);
  const size_t le = (size_t)n * 4 * H * W, ce = (size_t)n * L * 768, ue = (size_t)Lu * 768, re = (size_t)n * 3 * 64 * H * W;
  const size_t ne = step_noise ? ddim_timesteps(n_steps).size() * le : 0;
  float* d_c = (float*)c.io(0, ce * 4);
  float* d_u = (float*)c.io(1, ue * 4);
  float* d_l = init_latent ? (float*)c.io(2, le * 4) : nullptr;
  float* d_z = step_noise ? (float*)c.io(3, ne * 4) : nullptr;
  float* d_lo = latent_out ? (float*)c.io(4, le * 4) : nullptr;
  uint8_t* d_r = rgb ? (uint8_t*)c.io(5, re) : nullptr;
  SDB_CUDA(cudaMemcpyAsync(d_c, context, ce * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_u, uncond, ue * 4, cudaMemcpyHostToDevice, c.stream));
  if (init_latent) SDB_CUDA(cudaMemcpyAsync(d_l, init_latent, le * 4, cudaMemcpyHostToDevice, c.stream));
  if (step_noise) SDB_CUDA(cudaMemcpyAsync(d_z, step_noise, ne * 4, cudaMemcpyHostToDevice, c.stream));
  model_sample_ex_dev(c, d_c, n, L, d_u, Lu, scale, n_steps, sampler, eta, d_l, d_z, seed, H, W, d_lo, d_r, c.stream);
  if (latent_out) SDB_CUDA(cudaMemcpyAsync(latent_out, d_lo, le * 4, cudaMemcpyDeviceToHost, c.stream));
  if (rgb) SDB_CUDA(cudaMemcpyAsync(rgb, d_r, re, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

void model_randn_host(Ctx& c, uint64_t seed, int64_t count, float* out) {
  SDB_CHECK(count >= 0 && (out || count == 0), "randn: count must be >= 0 and out non-null");
  if (count == 0) return;
  float* d = (float*)c.io(0, (size_t)count * 4);
  randn_launch(d, (long long)count, seed, c.stream);
  SDB_CUDA(cudaMemcpyAsync(out, d, (size_t)count * 4, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

// ---- img2img (SDEdit) and latent-blend inpainting (DESIGN.md §7 row f5). The reference has no img2img: this is the standard
// construction on its own schedule and sampler (oracle/img2img_oracle.py states it once).
static void check_img2img_args(const uint8_t* rgb, const void* latent_out, const void* rgb_out, int n, int L, int Lu,
                               int n_steps, double strength, int H, int W) {
  SDB_CHECK(rgb, "img2img: rgb is null");
  SDB_CHECK(latent_out || rgb_out, "img2img: latent_out and rgb_out are both null");
  SDB_CHECK(strength >= 0.0 && strength <= 1.0, "img2img: strength must lie in [0, 1]");  // false for NaN
  check_sample_args(n, L, Lu, n_steps, H, W);
  check_encode_size(n, 8 * H, 8 * W);
}

// schedule index of the first step that runs: n_run = min(T, floor(strength * T + 1e-9)) of the T steps run, from T - n_run
static int img2img_start_index(int n_steps, double strength) {
  const int T = (int)ddim_timesteps(n_steps).size();
  return T - std::min(T, (int)std::floor(strength * T + 1e-9));
}

void model_img2img_dev(Ctx& c, const uint8_t* d_rgb_in, const uint8_t* d_mask, const float* d_context, int n, int L,
                       const float* d_uncond, int Lu, double scale, int n_steps, double strength, const float* d_noise,
                       uint64_t seed, int H, int W, float* d_latent_out, uint8_t* d_rgb, cudaStream_t caller) {
  check_img2img_args(d_rgb_in, d_latent_out, d_rgb, n, L, Lu, n_steps, strength, H, W);
  StreamJoin join(c, caller);
  const size_t le = (size_t)n * 4 * H * W;
  // x0, eps and the latent mask outlive the work-arena reset of the step loop: Ctx::state, not the work arena
  float* x0 = (float*)c.state(0, le * 4);
  const float* eps = d_noise;
  if (!d_noise) {
    float* e = (float*)c.state(1, le * 4);
    KernelScope ks(c, KC_ELEMENTWISE);
    randn_launch(e, (long long)le, seed, c.stream);  // the stream text-to-image draws its initial latent from
    eps = e;
  }
  uint8_t* lm = nullptr;
  if (d_mask) {
    lm = (uint8_t*)c.state(2, (size_t)n * H * W);
    KernelScope ks(c, KC_ELEMENTWISE);
    latent_mask_launch(d_mask, n, H, W, lm, c.stream);
  }
  // x0 = fl(encode_image(rgb * fl32(2/255) - 1) * 0.18215f), the inverse of latent_to_image's latent * (1 / 0.18215)
  c.work.reset();
  const size_t plane = (size_t)64 * H * W;
  for (int i0 = 0; i0 < n; i0 += 4) {  // chunks of 4 images, as model_encode_dev
    const int nb = std::min(4, n - i0);
    const size_t mark = c.work.off;
    float* img4 = c.work.get<float>((size_t)nb * 4 * plane);
    {
      KernelScope ks(c, KC_ELEMENTWISE);
      rgb8_to_planes4_launch(d_rgb_in + (size_t)i0 * 3 * plane, nb, 8 * H, 8 * W, img4, c.stream);
    }
    Fwd f(c, nb);
    vae_encode(f, img4, 8 * H, 8 * W, x0 + (size_t)i0 * 4 * H * W);
    c.work.off = mark;
  }
  {
    KernelScope ks(c, KC_ELEMENTWISE);
    scale_launch(x0, (long long)le, 0.18215f, c.stream);
  }
  const int i0 = img2img_start_index(n_steps, strength);
  const float* lat = x0;  // strength 0: nothing runs, the result is x0
  if (i0 < (int)ddim_timesteps(n_steps).size()) {
    SampleStart st;
    st.i0 = i0, st.x0 = x0, st.eps = eps, st.m = lm;
    lat = sample_loop(c, d_context, n, L, d_uncond, Lu, scale, n_steps, nullptr, st, H, W);
  }
  if (d_latent_out) SDB_CUDA(cudaMemcpyAsync(d_latent_out, lat, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  if (d_rgb) latent_to_image_dev(c, lat, n, H, W, d_rgb, d_rgb_in, d_mask);
}

void model_img2img_host(Ctx& c, const uint8_t* rgb_in, const uint8_t* mask, const float* context, int n, int L,
                        const float* uncond, int Lu, double scale, int n_steps, double strength, const float* noise, uint64_t seed,
                        int H, int W, float* latent_out, uint8_t* rgb) {
  check_img2img_args(rgb_in, latent_out, rgb, n, L, Lu, n_steps, strength, H, W);
  const size_t le = (size_t)n * 4 * H * W, ce = (size_t)n * L * 768, ue = (size_t)Lu * 768, re = (size_t)n * 3 * 64 * H * W;
  uint8_t* d_in = (uint8_t*)c.io(0, re);
  uint8_t* d_m = mask ? (uint8_t*)c.io(1, (size_t)n * 64 * H * W) : nullptr;
  float* d_c = (float*)c.io(2, ce * 4);
  float* d_u = (float*)c.io(3, ue * 4);
  float* d_n = noise ? (float*)c.io(4, le * 4) : nullptr;
  float* d_lo = latent_out ? (float*)c.io(5, le * 4) : nullptr;
  uint8_t* d_r = rgb ? (uint8_t*)c.io(6, re) : nullptr;
  SDB_CUDA(cudaMemcpyAsync(d_in, rgb_in, re, cudaMemcpyHostToDevice, c.stream));
  if (mask) SDB_CUDA(cudaMemcpyAsync(d_m, mask, (size_t)n * 64 * H * W, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_c, context, ce * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_u, uncond, ue * 4, cudaMemcpyHostToDevice, c.stream));
  if (noise) SDB_CUDA(cudaMemcpyAsync(d_n, noise, le * 4, cudaMemcpyHostToDevice, c.stream));
  model_img2img_dev(c, d_in, d_m, d_c, n, L, d_u, Lu, scale, n_steps, strength, d_n, seed, H, W, d_lo, d_r, c.stream);
  if (latent_out) SDB_CUDA(cudaMemcpyAsync(latent_out, d_lo, le * 4, cudaMemcpyDeviceToHost, c.stream));
  if (rgb) SDB_CUDA(cudaMemcpyAsync(rgb, d_r, re, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

void model_sample_host(Ctx& c, const float* context, int n, int L, const float* uncond, int Lu, double scale, int n_steps,
                       const float* init_latent, uint64_t seed, int H, int W, float* latent_out, uint8_t* rgb) {
  const size_t le = (size_t)n * 4 * H * W, ce = (size_t)n * L * 768, ue = (size_t)Lu * 768, re = (size_t)n * 3 * 64 * H * W;
  float* d_c = (float*)c.io(0, ce * 4);
  float* d_u = (float*)c.io(1, ue * 4);
  float* d_l = (float*)c.io(2, le * 4);
  float* d_lo = latent_out ? (float*)c.io(3, le * 4) : nullptr;
  uint8_t* d_r = rgb ? (uint8_t*)c.io(4, re) : nullptr;
  SDB_CUDA(cudaMemcpyAsync(d_c, context, ce * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_u, uncond, ue * 4, cudaMemcpyHostToDevice, c.stream));
  if (init_latent)
    SDB_CUDA(cudaMemcpyAsync(d_l, init_latent, le * 4, cudaMemcpyHostToDevice, c.stream));
  else
    randn_launch(d_l, (long long)le, seed, c.stream);
  model_sample_dev(c, d_c, n, L, d_u, Lu, scale, n_steps, d_l, H, W, d_lo, d_r, c.stream);
  if (latent_out) SDB_CUDA(cudaMemcpyAsync(latent_out, d_lo, le * 4, cudaMemcpyDeviceToHost, c.stream));
  if (rgb) SDB_CUDA(cudaMemcpyAsync(rgb, d_r, re, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

// forward_diffuser (stablediffusion/mod.rs:162-192): the two UNet evaluations of one guidance step as ONE batch-2n pass (the
// same pass sample_latent replays as a CUDA graph), then pred = u + (c - u) * scale. d_u / d_c may be null.
void model_forward_diffuser_dev(Ctx& c, const float* d_latent, int t, const float* d_context, int n, int L, const float* d_uncond,
                                int Lu, double scale, int H, int W, float* d_pred, float* d_u, float* d_c, cudaStream_t caller) {
  SDB_CHECK(n >= 1 && L >= 1 && Lu >= 1 && t >= 0 && t < 1000, "forward_diffuser arguments");
  SDB_CHECK(H % 8 == 0 && W % 8 == 0 && ((H / 8) * (W / 8)) % 8 == 0, "unsupported latent size");
  StreamJoin join(c, caller);
  c.work.reset();
  const int nb = 2 * n;
  const int Lpad = round_up(std::max(L, Lu), 32);
  const size_t le = (size_t)n * 4 * H * W;
  float* ctxp = c.work.get<float>((size_t)nb * Lpad * 768);
  float* xb = c.work.get<float>(2 * le);
  float* eps = c.work.get<float>(2 * le);
  int* d_t = c.work.get<int>(1);
  int* d_len = c.work.get<int>(nb);
  SDB_CUDA(cudaMemsetAsync(ctxp, 0, (size_t)nb * Lpad * 768 * 4, c.stream));
  for (int i = 0; i < n; ++i)
    SDB_CUDA(cudaMemcpyAsync(ctxp + (size_t)i * Lpad * 768, d_uncond, (size_t)Lu * 768 * 4, cudaMemcpyDeviceToDevice, c.stream));
  SDB_CUDA(cudaMemcpy2DAsync(ctxp + (size_t)n * Lpad * 768, (size_t)Lpad * 768 * 4, d_context, (size_t)L * 768 * 4,
                             (size_t)L * 768 * 4, n, cudaMemcpyDeviceToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(xb, d_latent, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(xb + le, d_latent, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  std::vector<int> lens(nb);
  for (int i = 0; i < nb; ++i) lens[i] = i < n ? Lu : L;
  SDB_CUDA(cudaMemcpyAsync(d_t, &t, 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_len, lens.data(), nb * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  unet_pass(c, nb, xb, d_t, ctxp, Lpad, d_len, H, W, eps, nullptr);
  if (d_u) SDB_CUDA(cudaMemcpyAsync(d_u, eps, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  if (d_c) SDB_CUDA(cudaMemcpyAsync(d_c, eps + le, le * 4, cudaMemcpyDeviceToDevice, c.stream));
  if (d_pred) {
    KernelScope ks(c, KC_ELEMENTWISE);
    cfg_combine_launch(eps, eps + le, (long long)le, (float)scale, d_pred, c.stream);
  }
}

void model_forward_diffuser_host(Ctx& c, const float* latent, int t, const float* context, int n, int L, const float* uncond,
                                 int Lu, double scale, int H, int W, float* pred, float* out_u, float* out_c) {
  const size_t le = (size_t)n * 4 * H * W, ce = (size_t)n * L * 768, ue = (size_t)Lu * 768;
  float* d_l = (float*)c.io(0, le * 4);
  float* d_c = (float*)c.io(1, ce * 4);
  float* d_u = (float*)c.io(2, ue * 4);
  float* d_o = (float*)c.io(3, 3 * le * 4);
  SDB_CUDA(cudaMemcpyAsync(d_l, latent, le * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_c, context, ce * 4, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(d_u, uncond, ue * 4, cudaMemcpyHostToDevice, c.stream));
  model_forward_diffuser_dev(c, d_l, t, d_c, n, L, d_u, Lu, scale, H, W, d_o, d_o + le, d_o + 2 * le, c.stream);
  if (pred) SDB_CUDA(cudaMemcpyAsync(pred, d_o, le * 4, cudaMemcpyDeviceToHost, c.stream));
  if (out_u) SDB_CUDA(cudaMemcpyAsync(out_u, d_o + le, le * 4, cudaMemcpyDeviceToHost, c.stream));
  if (out_c) SDB_CUDA(cudaMemcpyAsync(out_c, d_o + 2 * le, le * 4, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

// ================================================================================ CLIP text encoder
// reference src/model/clip/mod.rs:56-75 (CLIP::forward), :109-115 (block), :158-180 (attention with the causal mask of
// src/backend.rs:130-139), :204-227 (MLP with QuickGELU). tokens [n][L] int32 -> out [n][L][768]. SURVEY §8f row f1.
void model_clip_forward_dev(Ctx& c, const int* d_tok, int n, int L, float* d_out, cudaStream_t caller) {
  Model& m = M(c);
  SDB_CHECK(n >= 1 && L >= 1 && L <= 77, "clip_forward: 1 <= L <= 77 (position table), n >= 1");
  StreamJoin join(c, caller);
  c.work.reset();
  Fwd f(c, n);
  const int D = 768, heads = 12;
  const int Lp = round_up(L, 8);           // per-sample row pitch: keeps every TMA tile origin 16-byte aligned
  const int Mr = n * Lp, Mp = round_up(Mr, 32);
  float* x = c.work.get<float>((size_t)Mr * D);
  float* y = c.work.get<float>((size_t)Mr * D);
  Half2Ptr l16 = f.half2((size_t)Mr * D, true), o16 = f.half2((size_t)Mr * D, true), h16 = f.half2((size_t)Mr * 4 * D, true);
  __half* qk = c.work.get<__half>((size_t)Mr * 2 * D);
  __half* vT = c.work.get<__half>((size_t)D * Mp);
  // pad rows (l >= L) never reach a real row (causal mask, row-wise ops) but must stay finite: 0 * NaN would poison P.V
  SDB_CUDA(cudaMemsetAsync(o16.hi, 0, (size_t)Mr * D * 2, c.stream));
  SDB_CUDA(cudaMemsetAsync(o16.lo, 0, (size_t)Mr * D * 2, c.stream));
  {
    KernelScope ks(c, KC_ELEMENTWISE);
    embed_tokens_launch(d_tok, mptr(c, m.clip.tok_i), mptr(c, m.clip.pos_i), n, L, Lp, D, 49408, x, c.stream);
  }
  auto ln = [&](const NormW& nw, Half2Ptr o, float* o32) {
    KernelScope ks(c, KC_LAYERNORM);
    layernorm_launch(x, Mr, D, nw.gamma, nw.beta, nw.eps, o, o32, c.stream);
  };
  for (ClipBlockW& cb : m.clip.blocks) {
    ln(cb.attn_ln, l16, nullptr);
    {
      Epilogue ep;
      ep.out_f16.hi = qk, ep.bias = cb.bias_qk;
      run_gemm(c, G_LINEAR, f.rows_operand(l16, Mr, D), nullptr, cb.w_qk, 3, ep);
    }
    {
      WeightOp tok;
      tok.p = l16, tok.N = Mp, tok.rows = Mr, tok.K = D;
      Epilogue ep;
      ep.out_f16.hi = vT;
      run_gemm(c, G_LINEAR, f.rows_operand(cb.value.packed.p, D, D), nullptr, tok, 3, ep);
    }
    {
      AttnOp at;
      at.q = qk, at.ldq = 2 * D, at.q_col0 = 0, at.q_rows = Lp;
      at.k = qk, at.ldk = 2 * D, at.k_col0 = D, at.k_rows = Lp;
      at.vT = vT, at.ldv = Mp;
      at.nb = n, at.heads = heads, at.d = 64, at.dpad = 64, at.Nq = L, at.Nk = L;
      at.causal = 1;
      at.out = o16, at.ldo = D;
      run_attention(c, at);
    }
    {
      Epilogue ep;
      ep.out_f32 = x, ep.residual = x, ep.bias = cb.bias_out;
      run_gemm(c, G_LINEAR, f.rows_operand(o16, Mr, D), nullptr, cb.out.packed, 3, ep);
    }
    ln(cb.mlp_ln, l16, nullptr);
    {
      Epilogue ep;
      ep.out_f16 = h16, ep.bias = cb.fc1.bias, ep.act = 1;
      run_gemm(c, G_LINEAR, f.rows_operand(l16, Mr, D), nullptr, cb.fc1.packed, 3, ep);
    }
    {
      Epilogue ep;
      ep.out_f32 = x, ep.residual = x, ep.bias = cb.fc2.bias;
      run_gemm(c, G_LINEAR, f.rows_operand(h16, Mr, 4 * D), nullptr, cb.fc2.packed, 3, ep);
    }
  }
  ln(m.clip.ln_final, Half2Ptr{}, y);
  SDB_CUDA(cudaMemcpy2DAsync(d_out, (size_t)L * D * 4, y, (size_t)Lp * D * 4, (size_t)L * D * 4, n, cudaMemcpyDeviceToDevice,
                             c.stream));
}

void model_clip_forward_host(Ctx& c, const int* tokens, int n, int L, float* out) {
  SDB_CHECK(n >= 1 && L >= 1 && L <= 77, "clip_forward: 1 <= L <= 77 (position table), n >= 1");
  // the reference's embedding lookup panics on an id outside the table; the host entry rejects it (the *_dev entry,
  // which cannot see the ids without a sync, clamps instead)
  for (long long i = 0; i < (long long)n * L; ++i)
    SDB_CHECK(tokens[i] >= 0 && tokens[i] < 49408, "clip_forward: token id outside the 49408-entry vocabulary");
  int* d_t = (int*)c.io(0, (size_t)n * L * 4);
  float* d_o = (float*)c.io(1, (size_t)n * L * 768 * 4);
  SDB_CUDA(cudaMemcpyAsync(d_t, tokens, (size_t)n * L * 4, cudaMemcpyHostToDevice, c.stream));
  model_clip_forward_dev(c, d_t, n, L, d_o, c.stream);
  SDB_CUDA(cudaMemcpyAsync(out, d_o, (size_t)n * L * 768 * 4, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
}

// ================================================================================ attention unit-test entry
void model_test_attention(Ctx& c, const float* q, const float* k, const float* v, int n, int Nq, int Nk, int C, int heads,
                          float* out) {
  // stages q / k|v exactly as the SpatialTransformer does: head-padded rows, V row-major beside K (consumed MN-major)
  const int d = C / heads, dpad = (d % 16 == 0) ? d : (d + 15) / 16 * 16, hd = heads * dpad;
  const int Nkp = round_up(Nk, 8);
  std::vector<__half> hq((size_t)n * Nq * hd, __float2half(0.f)), hkv((size_t)n * Nkp * 2 * hd, __float2half(0.f));
  std::vector<__half> hq_lo(hq.size(), __float2half(0.f)), hkv_lo(hkv.size(), __float2half(0.f));
  auto split = [](float v, __half& hi, __half& lo) {
    hi = __float2half(v);
    lo = __float2half(v - __half2float(hi));
  };
  for (int s = 0; s < n; ++s)
    for (int i = 0; i < Nq; ++i)
      for (int h = 0; h < heads; ++h)
        for (int j = 0; j < d; ++j)
          split(q[((size_t)s * Nq + i) * C + h * d + j], hq[((size_t)s * Nq + i) * hd + h * dpad + j], hq_lo[((size_t)s * Nq + i) * hd + h * dpad + j]);
  for (int s = 0; s < n; ++s)
    for (int i = 0; i < Nk; ++i)
      for (int h = 0; h < heads; ++h)
        for (int j = 0; j < d; ++j) {
          split(k[((size_t)s * Nk + i) * C + h * d + j], hkv[((size_t)s * Nkp + i) * 2 * hd + h * dpad + j], hkv_lo[((size_t)s * Nkp + i) * 2 * hd + h * dpad + j]);
          hkv[((size_t)s * Nkp + i) * 2 * hd + hd + h * dpad + j] = __float2half(v[((size_t)s * Nk + i) * C + h * d + j]);
        }
  __half* dq = c.work.get<__half>(hq.size());
  __half* dkv = c.work.get<__half>(hkv.size());
  __half* dq_lo = c.work.get<__half>(hq.size());
  __half* dkv_lo = c.work.get<__half>(hkv.size());
  SDB_CUDA(cudaMemcpyAsync(dq_lo, hq_lo.data(), hq.size() * 2, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(dkv_lo, hkv_lo.data(), hkv.size() * 2, cudaMemcpyHostToDevice, c.stream));
  Half2Ptr o16;
  o16.hi = c.work.get<__half>((size_t)n * Nq * C);
  o16.lo = c.work.get<__half>((size_t)n * Nq * C);
  int* dlen = c.work.get<int>(n);
  std::vector<int> lens(n, Nk);
  SDB_CUDA(cudaMemcpyAsync(dq, hq.data(), hq.size() * 2, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(dkv, hkv.data(), hkv.size() * 2, cudaMemcpyHostToDevice, c.stream));
  SDB_CUDA(cudaMemcpyAsync(dlen, lens.data(), n * 4, cudaMemcpyHostToDevice, c.stream));
  AttnOp at;
  at.q = dq, at.ldq = hd, at.q_rows = Nq;
  at.k = dkv, at.ldk = 2 * hd, at.k_rows = Nkp;
  at.vT = dkv, at.ldv = 2 * hd, at.v_mn = 1, at.v_col0 = hd;
  at.q_lo = dq_lo, at.k_lo = dkv_lo;  // used by the head dims that have the split-product kernel (40, 80) unless attn_split = 0
  at.nb = n, at.heads = heads, at.d = d, at.dpad = dpad, at.Nq = Nq, at.Nk = Nkp;
  at.kvlen = dlen;
  at.out = o16, at.ldo = C;
  run_attention(c, at);
  std::vector<__half> hi((size_t)n * Nq * C), lo((size_t)n * Nq * C);
  SDB_CUDA(cudaMemcpyAsync(hi.data(), o16.hi, hi.size() * 2, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaMemcpyAsync(lo.data(), o16.lo, lo.size() * 2, cudaMemcpyDeviceToHost, c.stream));
  SDB_CUDA(cudaStreamSynchronize(c.stream));
  for (size_t i = 0; i < hi.size(); ++i) out[i] = __half2float(hi[i]) + __half2float(lo[i]);
}

}  // namespace sdb
