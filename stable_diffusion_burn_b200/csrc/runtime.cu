// runtime.cu — context plumbing, TMA tensor maps and the GEMM op builder.
#include "runtime.cuh"

#include <algorithm>

#include <cudaTypedefs.h>

#include <cmath>
#include <cstdlib>
#include <cstring>

namespace sdb {

// Programmatic dependent launch (measured, tools/step_time.py, one process): off 155.3 ms/image; on with every kernel releasing its
// dependents at entry 155.3 -> +1 % (early CTAs of the next kernel sit on the SMs while the GEMM still runs); on with the GEMMs
// releasing them when their epilogue starts and loading their first weight tiles ahead of griddepcontrol.wait: -2.3 %.
// SDB_PDL=0 disables, 1 = release at entry everywhere, 2 (default) = late release in the GEMMs.
int g_pdl_late = 1;
bool g_pdl_enabled = true;

// ------------------------------------------------------------------ arena
void Arena::init(size_t bytes) {
  SDB_CUDA(cudaMalloc(&base, bytes));
  cap = bytes;
  off = 0;
}
void Arena::destroy() {
  if (base) cudaFree(base);
  base = nullptr;
  cap = off = 0;
}
void* Arena::alloc(size_t bytes) {
  const size_t a = (off + 1023) & ~size_t(1023);
  if (a + bytes > cap)
    throw Error("arena exhausted: need " + std::to_string(a + bytes) + " of " + std::to_string(cap) + " bytes");
  off = a + bytes;
  if (off > high) high = off;
  return base + a;
}

static void* grow(Ctx::IoBuf& b, size_t bytes, cudaStream_t stream) {
  if (bytes > b.cap) {
    SDB_CUDA(cudaStreamSynchronize(stream));  // nothing queued may still read the old buffer
    if (b.p) cudaFree(b.p);
    b.p = nullptr, b.cap = 0;
    const size_t want = (bytes + (1u << 20) - 1) & ~size_t((1u << 20) - 1);
    SDB_CUDA(cudaMalloc(&b.p, want));
    b.cap = want;
  }
  return b.p;
}
void* Ctx::io(int slot, size_t bytes) { return grow(iobuf[slot], bytes, stream); }
void* Ctx::state(int slot, size_t bytes) { return grow(statebuf[slot], bytes, stream); }
void Ctx::io_destroy() {
  for (IoBuf* set : {iobuf, statebuf})
    for (int i = 0; i < 8; ++i) {
      IoBuf& b = set[i];
      if (b.p) cudaFree(b.p);
      b.p = nullptr, b.cap = 0;
    }
}

float* Ctx::master_ptr(const std::string& name) {
  auto it = index.find(name);
  if (it == index.end()) throw Error("unknown tensor: " + name);
  return reinterpret_cast<float*>(master.base) + tensors[it->second].offset;
}
const TensorInfo& Ctx::info(const std::string& name) {
  auto it = index.find(name);
  if (it == index.end()) throw Error("unknown tensor: " + name);
  return tensors[it->second];
}

const char* kernel_class_name(int cls) {
  static const char* names[KC_COUNT] = {"gemm_tc", "splitk_reduce", "attention", "gn_stats", "prep_operand",
                                        "layernorm", "small_conv", "elementwise"};
  return (cls >= 0 && cls < KC_COUNT) ? names[cls] : "?";
}

// ------------------------------------------------------------------ profiling scope
KernelScope::KernelScope(Ctx& c_, int cls_, double flops, double bytes, double issued) : c(c_), cls(cls_), on(c_.profiling) {
  c.launches++;
  c.cls_launches[cls]++;
  c.cls_flops[cls] += flops;
  c.cls_bytes[cls] += bytes;
  c.cls_issued[cls] += issued;
  static FILE* label_log = getenv("SDB_LABEL_LOG") ? fopen(getenv("SDB_LABEL_LOG"), "w") : nullptr;  // launch-order labels (ncu join)
  if (label_log) fprintf(label_log, "%s\t%s\n", kernel_class_name(cls), c.dbg_label.c_str()), fflush(label_log);
  if (on) {
    ev.cls = cls;
    ev.flops = flops;
    ev.bytes = bytes;
    ev.label = c.dbg_label;
    cudaEventCreate(&ev.a);
    cudaEventCreate(&ev.b);
    cudaEventRecord(ev.a, c.stream);
  }
}
KernelScope::~KernelScope() {
  if (on) {
    cudaEventRecord(ev.b, c.stream);
    c.prof.push_back(ev);
  }
  if (c.debug_sync) {
    cudaError_t e = cudaStreamSynchronize(c.stream);
    if (e != cudaSuccess) {
      fprintf(stderr, "[sdb200] launch #%lld (%s) failed: %s | %s\n", (long long)c.launches, kernel_class_name(cls),
              cudaGetErrorString(e), c.dbg_label.c_str());
      fflush(stderr);
    }
  }
  c.dbg_label.clear();
}
void profile_collect(Ctx& c) {
  if (c.prof.empty()) return;
  cudaStreamSynchronize(c.stream);
  FILE* dump = getenv("SDB_PROFILE_DUMP") ? fopen(getenv("SDB_PROFILE_DUMP"), "a") : nullptr;
  for (auto& e : c.prof) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e.a, e.b);
    c.cls_ms[e.cls] += ms;
    if (dump) fprintf(dump, "%s\t%.3f\t%.4g\t%.4g\t%s\n", kernel_class_name(e.cls), ms * 1e3, e.flops, e.bytes, e.label.c_str());
    cudaEventDestroy(e.a);
    cudaEventDestroy(e.b);
  }
  if (dump) fclose(dump);
  c.prof.clear();
}

// ------------------------------------------------------------------ tensor maps
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    void* p = nullptr;
    SDB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (!p || qres != cudaDriverEntryPointSuccess) throw Error("cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// fp16 tensor [N][P][H][W][C]; box {64, bw, bh, 1, bn}; 128B swizzle; zero fill outside
static CUtensorMap make_act_map(const __half* ptr, int C, int W, int H, int P, int N, int bw, int bh, int bn) {
  CUtensorMap m;
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)P, (cuuint64_t)N};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2,
                           (cuuint64_t)P * H * W * C * 2};
  cuuint32_t box[5] = {64, (cuuint32_t)bw, (cuuint32_t)bh, 1, (cuuint32_t)bn};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<__half*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error("cuTensorMapEncodeTiled(act) failed: " + std::to_string((int)r));
  return m;
}
// fp16 matrix [rows][K]; box {64, brows}
static CUtensorMap make_w_map(const __half* ptr, int K, int rows, int brows, long long ld = 0) {
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(ld ? ld : K) * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)brows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error("cuTensorMapEncodeTiled(weight) failed: " + std::to_string((int)r));
  return m;
}

// plain fp16 matrix [rows][ld] with a {64, brows} box
static CUtensorMap make_mat_map(const __half* ptr, long long ld, long long rows, int brows) {
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)brows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error("cuTensorMapEncodeTiled(matrix) failed: " + std::to_string((int)r));
  return m;
}

void run_attention(Ctx& c, const AttnOp& a) {
  SDB_CHECK(a.ldq % 8 == 0 && a.ldk % 8 == 0 && a.ldv % 8 == 0, "attention leading dims must be multiples of 8");
  // the causal mask is applied inside the first key tile only (CLIP: L <= 77); longer causal sequences are not supported
  SDB_CHECK(!a.causal || a.Nk <= 128, "causal attention supports at most 128 keys");
  SDB_CHECK(a.Nk >= 1 && a.Nq >= 1, "attention needs at least one query and one key");
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.nb = a.nb, p.heads = a.heads, p.d = a.d, p.dpad = a.dpad, p.Nq = a.Nq, p.Nk = a.Nk;
  p.q_rows_per_sample = a.q_rows, p.k_rows_per_sample = a.k_rows;
  p.q_col0 = a.q_col0, p.k_col0 = a.k_col0;
  p.v_mn = a.v_mn, p.v_col0 = a.v_col0;
  p.kvlen = a.kvlen;
  p.causal = a.causal;
  p.scale = (float)(1.0 / std::sqrt((double)a.d));
  p.out_hi = a.out.hi, p.out_lo = a.out.lo, p.ldo = a.ldo;
  AttnMaps am;
  am.q = make_mat_map(a.q, a.ldq, (long long)a.nb * a.q_rows, 128);
  am.k = make_mat_map(a.k, a.ldk, (long long)a.nb * a.k_rows, 128);
  am.v = a.v_mn ? make_mat_map(a.vT, a.ldv, (long long)a.nb * a.k_rows, 128)
                : make_mat_map(a.vT, a.ldv, (long long)a.heads * a.d, a.dpad);
  p.qk3 = (a.q_lo && a.k_lo && a.v_mn && attention_supports_qk3(a.dpad) && c.opt_attn_split) ? 1 : 0;
  am.q_lo = p.qk3 ? make_mat_map(a.q_lo, a.ldq, (long long)a.nb * a.q_rows, 128) : am.q;
  am.k_lo = p.qk3 ? make_mat_map(a.k_lo, a.ldk, (long long)a.nb * a.k_rows, 128) : am.k;
  const double flops = 4.0 * a.nb * a.heads * (double)a.Nq * a.Nk * a.d;  // algorithmic (the split QK^T issues 2x this)
  if (c.debug_sync || c.profiling || getenv("SDB_LABEL_LOG")) {
    char buf[200];
    snprintf(buf, sizeof(buf), "attention nb=%d heads=%d d=%d dpad=%d Nq=%d Nk=%d ldq=%d ldk=%d ldv=%d kvlen=%p", a.nb, a.heads,
             a.d, a.dpad, a.Nq, a.Nk, a.ldq, a.ldk, a.ldv, (const void*)a.kvlen);
    c.dbg_label = buf;
  }
  static const bool dbg_on = getenv("SDB_ATTN_DBG") != nullptr;
  static long long* dbg_buf = nullptr;
  if (dbg_on) {
    if (!dbg_buf) SDB_CUDA(cudaMallocManaged(&dbg_buf, 256 * sizeof(long long)));
    SDB_CUDA(cudaStreamSynchronize(c.stream));
    memset(dbg_buf, 0, 256 * sizeof(long long));
    p.dbg = dbg_buf;
  }
  {
    KernelScope ks(c, KC_ATTN, flops, 0);
    attention_launch(am, p, c.stream);
  }
  if (dbg_on) {  // bring-up aid: per-key-tile timeline of CTA (0,0,0), cycles since kernel entry
    SDB_CUDA(cudaStreamSynchronize(c.stream));
    const long long t0 = dbg_buf[255];
    auto rel = [&](int i) { return dbg_buf[i] ? dbg_buf[i] - t0 : -1; };
    fprintf(stderr, "attn_dbg nb=%d d=%d Nq=%d Nk=%d qk3=%d\n", a.nb, a.d, a.Nq, a.Nk, p.qk3);
    for (int jj = 0; jj < 4; ++jj) {
      for (int g = 0; g < 2; ++g)
        fprintf(stderr, "  j=%d softmax g%d: wait_s %lld s_ready %lld loaded %lld max %lld pv_ok %lld rescaled %lld exps %lld p_arrive %lld\n", 8 + jj, g,
                rel(g * 64 + jj * 8 + 0), rel(g * 64 + jj * 8 + 1), rel(g * 64 + jj * 8 + 2), rel(g * 64 + jj * 8 + 3), rel(g * 64 + jj * 8 + 4),
                rel(g * 64 + jj * 8 + 5), rel(g * 64 + jj * 8 + 6), rel(g * 64 + jj * 8 + 7));
      for (int g = 0; g < 2; ++g)
        fprintf(stderr, "  j=%d mma g%d: qk(j+1) begin %lld k_ok %lld issued %lld | pv: v_ok %lld p_ok %lld issued %lld\n", 8 + jj, g,
                rel(128 + jj * 16 + g * 8 + 0), rel(128 + jj * 16 + g * 8 + 4), rel(128 + jj * 16 + g * 8 + 1), rel(128 + jj * 16 + g * 8 + 5),
                rel(128 + jj * 16 + g * 8 + 2), rel(128 + jj * 16 + g * 8 + 3));
    }
  }
}

static int pow2_floor(int x) {
  int p = 1;
  while (p * 2 <= x) p *= 2;
  return p;
}
static int pow2_ceil(int x) {
  int p = 1;
  while (p < x) p *= 2;
  return p;
}

// ------------------------------------------------------------------ GEMM op
void run_gemm(Ctx& c, int kind, const ActOp& a0in, const ActOp* a1in, const WeightOp& w, int passes, const Epilogue& ep,
              const ExtraK* xk) {
  ActOp a0 = a0in, a1;
  if (a1in) a1 = *a1in;
  int gn_rpi = ep.gn_rpi, gn_nimg = 0;
  if (kind == G_CONV1) {  // a 1x1 conv over NHWC is a plain row-major GEMM
    gn_rpi = a0.H * a0.W;
    a0.W = a0.n * a0.H * a0.W, a0.H = 1, a0.n = 1;
    if (a1in) a1.W = a1.n * a1.H * a1.W, a1.H = 1, a1.n = 1;
    kind = G_LINEAR;
  }
  SDB_CHECK(a0.C % 64 == 0, "A channels must be a multiple of 64");
  SDB_CHECK(!a1in || a1.C % 64 == 0, "A1 channels must be a multiple of 64");
  if (c.opt_precision >= 1 && c.opt_precision <= 3) passes = c.opt_precision;
  SDB_CHECK(passes >= 1 && passes <= 3, "passes");
  SDB_CHECK(passes < 2 || a0.p.lo, "multi-pass GEMM needs the lo half of A");
  SDB_CHECK(passes < 2 || !a1in || a1.p.lo, "multi-pass GEMM needs the lo half of A1");
  SDB_CHECK(passes < 3 || w.p.lo, "3-pass GEMM needs the lo half of W");

  GemmParams p;
  memset(&p, 0, sizeof(p));
  const int Ctot = a0.C + (a1in ? a1.C : 0);
  p.nimg = a0.n, p.H = a0.H, p.W = a0.W;
  p.N = w.N;
  p.kc = Ctot / 64;
  p.kc0 = a0.C / 64;
  int phases_out = 1;
  switch (kind) {
    case G_LINEAR:
      p.num_taps = 1;
      break;
    case G_CONV3:
      p.num_taps = 9;
      for (int t = 0; t < 9; ++t) p.tap_dh[t] = t / 3 - 1, p.tap_dw[t] = t % 3 - 1, p.tap_ph[t] = 0;
      break;
    case G_CONV3_S2:
      SDB_CHECK(a0.P == 4, "stride-2 conv needs a 4-phase operand");
      p.num_taps = 9;
      for (int t = 0; t < 9; ++t) {
        const int kh = t / 3, kw = t % 3;
        p.tap_dh[t] = kh == 0 ? -1 : 0;
        p.tap_dw[t] = kw == 0 ? -1 : 0;
        p.tap_ph[t] = (kh != 1 ? 2 : 0) + (kw != 1 ? 1 : 0);
      }
      break;
    case G_CONV3_S2_PAD01:
      // input row 2y + kh: kh = 0 even row y, kh = 1 odd row y, kh = 2 even row y + 1 (row H is the zero pad: TMA OOB fill)
      SDB_CHECK(a0.P == 4, "stride-2 conv needs a 4-phase operand");
      p.num_taps = 9;
      for (int t = 0; t < 9; ++t) {
        const int kh = t / 3, kw = t % 3;
        p.tap_dh[t] = kh == 2 ? 1 : 0;
        p.tap_dw[t] = kw == 2 ? 1 : 0;
        p.tap_ph[t] = (kh == 1 ? 2 : 0) + (kw == 1 ? 1 : 0);
      }
      break;
    case G_CONV3_UP2:
      p.num_taps = 4;
      phases_out = 4;
      break;
    default:
      throw Error("bad gemm kind");
  }
  SDB_CHECK(w.K == p.num_taps * Ctot, "weight K does not match the operand");
  if (xk) {
    const int xC = xk->x0.C + (xk->has_x1 ? xk->x1.C : 0);
    SDB_CHECK(kind == G_CONV3 || kind == G_LINEAR, "extra-K operands need an unshifted output grid");
    SDB_CHECK(xk->x0.n == a0.n && xk->x0.H == a0.H && xk->x0.W == a0.W && xk->x0.P == 1 && xk->x0.C % 64 == 0, "extra-K geometry");
    SDB_CHECK(!xk->has_x1 || (xk->x1.n == a0.n && xk->x1.H == a0.H && xk->x1.W == a0.W && xk->x1.C % 64 == 0), "extra-K geometry");
    SDB_CHECK(xk->w.N == w.N && xk->w.K == xC, "extra-K weights");
    SDB_CHECK(passes < 2 || (xk->x0.p.lo && (!xk->has_x1 || xk->x1.p.lo)), "multi-pass GEMM needs the lo half of the extra operands");
    SDB_CHECK(passes < 3 || xk->w.p.lo, "3-pass GEMM needs the lo half of the extra weights");
    p.xkc0 = xk->x0.C / 64, p.xkc = xC / 64;
  }

  // M tile = TN x TH x TW output pixels
  p.TW = std::min(pow2_floor(a0.W), 128);
  p.TH = std::min(128 / p.TW, pow2_ceil(a0.H));
  p.TN = 128 / (p.TW * p.TH);
  p.tiles_w = (a0.W + p.TW - 1) / p.TW;
  p.tiles_h = (a0.H + p.TH - 1) / p.TH;
  p.tiles_n = (a0.n + p.TN - 1) / p.TN;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;

  // CTA pairs along M issue one cta_group::2 MMA (256 x BN): each CTA stages only half of the weight tile.
  // Needs an even number of M tiles and no split-K (decided below).
  bool pair = c.opt_cluster && (m_tiles % 2 == 0);
  // N tile (measured per layer in profiles/r1_gemm_layers.md): 160 divides the UNet widths 320/640/1280 evenly
  int BN;
  if (ep.geglu)
    BN = 128;
  else if (pair && c.opt_pair_bn256 && w.N % 256 == 0 && (long long)m_tiles * (w.N / 256) >= 64)
    BN = 256;  // pair tile 256 x 256: the fewest operand bytes per FLOP
  else if (w.N % 160 == 0)
    BN = 160;
  else if (w.N % 256 == 0 && (long long)m_tiles * (w.N / 256) >= 296)
    BN = 256;
  else if (w.N % 128 == 0)
    BN = 128;
  else
    BN = 64;
  if (ep.ln_out) {
    SDB_CHECK(w.N % 160 == 0 && !ep.geglu, "LayerNorm statistics need an output width that tiles by 160");
    BN = 160;
  }
  if (ep.ln_in) SDB_CHECK(BN == 128 || BN == 160, "LayerNorm-consuming GEMM: tile width");
  const int n_tiles = (w.N + BN - 1) / BN;


  // split-K when the grid cannot fill the machine and the K loop is long
  const int iters = p.num_taps * p.kc + p.xkc;
  int split = 1;
  if (c.opt_splitk && kind != G_CONV3_UP2 && !ep.geglu && !ep.ln_out && !ep.ln_in) {
    const int ctas = m_tiles * n_tiles;
    if (ctas <= 74 && iters >= c.opt_splitk_min_iters) {
      // floor: ctas*split must stay within ONE wave of the 148 SMs (a 2-wave grid costs 2x, see profiles/r1);
      // every split keeps >= 16 k-chunks so the rendezvous + fold stays small against its mainloop
      split = std::min(std::min(148 / ctas, iters / c.opt_splitk_chunk), 16);
      if (split < 1) split = 1;
    }
  }
  p.cluster = pair ? 2 : 1;  // pairs and split-K compose: a cluster spans x only, both CTAs share blockIdx.z
  if (split > 1) {  // no empty K ranges: every split must own at least one iteration
    const int per = (iters + split - 1) / split;
    split = (iters + per - 1) / per;
  }
  p.split_k = split;
  static const bool gemm_dbg = getenv("SDB_GEMM_DBG") != nullptr || getenv("SDB_LABEL_LOG") != nullptr;
  if (c.debug_sync || c.profiling || gemm_dbg) {
    char buf[256];
    snprintf(buf, sizeof(buf), "gemm kind=%d n=%d H=%d W=%d P=%d C0=%d C1=%d N=%d K=%d xk=%d BN=%d split=%d passes=%d geglu=%d epi=%s%s tile=%dx%dx%d cluster=%d",
             kind, a0.n, a0.H, a0.W, a0.P, a0.C, a1in ? a1.C : 0, w.N, w.K, p.xkc * 64, BN, split, passes, ep.geglu,
             ep.gn ? "gn" : (ep.ln_out ? "lns" : (ep.ln_in ? "lnc" : "-")), ep.residual16.hi ? "+r16" : (ep.residual ? "+r32" : ""), p.TN, p.TH, p.TW, p.cluster);
    c.dbg_label = buf;
  }

  // GroupNorm statistics of the output: needs every 32-row lane quarter inside one image, buckets that tile BN, slot room
  GnPart* gn = ep.gn;
  if (gn) {
    int slots = m_tiles / p.tiles_n * split * phases_out;
    bool geom = p.TN <= 4;
    if (kind == G_LINEAR && gn_rpi > 0) {  // rows are tokens of gn_nimg images, gn_rpi rows each
      const long long rows = (long long)a0.W;
      geom = rows % gn_rpi == 0 && (gn_rpi % 128 == 0 || (128 % gn_rpi == 0 && gn_rpi >= 32));
      gn_nimg = (int)(rows / gn_rpi);
      slots = (gn_rpi >= 128 ? gn_rpi / 128 : 1) * split;
    } else {
      if (kind == G_LINEAR) geom = false;  // rows without an image size: the caller must say how many rows make an image
      gn_rpi = 0;
    }
    const bool ok = gn->buf && gn->bucket > 0 && !ep.geglu && geom && BN >= 128 && BN % gn->bucket == 0 && w.N % gn->bucket == 0 &&
                    slots <= gn->cap && c.opt_gn_epilogue;
    gn->slots = ok ? slots : 0;
    if (!ok) gn = nullptr;
  }
  p.gn_part = gn ? gn->buf : nullptr;
  p.gn_cap = gn ? gn->cap : 0, p.gn_bucket = gn ? gn->bucket : 1;
  p.gn_rpi = gn ? gn_rpi : 0, p.gn_nimg = gn_nimg;
  p.ln_out = ep.ln_out, p.ln_slots = ln_slots(w.N);
  p.ln_in = ep.ln_in, p.ln_in_slots = ep.ln_in_slots, p.ln_C = ep.ln_C, p.ln_eps = ep.ln_eps;
  p.ln_u = passes >= 3 ? ep.ln_u_full : ep.ln_u_hi;
  SDB_CHECK(!ep.ln_in || (p.ln_u && ep.ln_in_slots > 0 && ep.ln_C == w.K && kind == G_LINEAR), "LayerNorm-consuming GEMM: arguments");
  SDB_CHECK(!ep.ln_in || (!ep.residual && !ep.rowbias && !ep.residual16.hi), "LayerNorm-consuming GEMM: no residual / row bias");
  SDB_CHECK(!ep.ln_out || kind == G_LINEAR, "LayerNorm statistics: rows must be tokens");
  p.res_hi = ep.residual16.hi, p.res_lo = ep.residual16.lo;
  SDB_CHECK(!ep.residual16.hi || (ep.residual16.lo && !ep.residual && !ep.rowbias), "fp16-pair residual: needs both halves, excludes the fp32 residual / row bias");
  p.out_f32 = ep.out_f32;
  p.out_f16 = ep.out_f16.hi;
  p.out_f16_lo = ep.out_f16.lo;
  p.bias = ep.bias;
  p.rowbias = ep.rowbias;
  p.residual = ep.residual;
  p.geglu = ep.geglu;
  p.act = ep.act;
  p.pdl_late = g_pdl_late;
  p.prefetch_w = (g_pdl_enabled && c.opt_prefetch_w && m_tiles <= 4) ? 1 : 0;
  const int nout = ep.geglu ? w.N / 2 : w.N;
  p.ldc = ep.ldc ? ep.ldc : nout;
  p.ldc16 = ep.ldc16 ? ep.ldc16 : nout;
  SDB_CHECK(!(ep.rowbias && ep.residual), "epilogue takes a time-embedding row or a residual, not both");
  p.os = (kind == G_CONV3_UP2) ? 2 : 1;
  p.OH = a0.H * p.os, p.OW = a0.W * p.os;
  SDB_CHECK((double)a0.n * p.OH * p.OW * (double)std::max(p.ldc, p.ldc16) < 2147483648.0,
            "GEMM output exceeds 2^31 elements (the epilogue uses 32-bit element offsets)");

  GemmMaps maps;
  memset(&maps, 0, sizeof(maps));
  maps.a[0][0] = make_act_map(a0.p.hi, a0.C, a0.W, a0.H, a0.P, a0.n, p.TW, p.TH, p.TN);
  maps.a[0][1] = maps.a[0][0];
  if (passes >= 2) maps.a[0][1] = make_act_map(a0.p.lo, a0.C, a0.W, a0.H, a0.P, a0.n, p.TW, p.TH, p.TN);
  maps.a[1][0] = maps.a[0][0];
  maps.a[1][1] = maps.a[0][1];
  if (a1in) {
    SDB_CHECK(a1.n == a0.n && a1.H == a0.H && a1.W == a0.W && a1.P == a0.P, "concat operand geometry");
    maps.a[1][0] = make_act_map(a1.p.hi, a1.C, a1.W, a1.H, a1.P, a1.n, p.TW, p.TH, p.TN);
    maps.a[1][1] = maps.a[1][0];
    if (passes >= 2) maps.a[1][1] = make_act_map(a1.p.lo, a1.C, a1.W, a1.H, a1.P, a1.n, p.TW, p.TH, p.TN);
  }

  for (int sidx = 2; sidx < 4; ++sidx) maps.a[sidx][0] = maps.a[sidx][1] = maps.a[0][0];
  if (xk) {
    auto xmaps = [&](const ActOp& x, int sidx) {
      maps.a[sidx][0] = make_act_map(x.p.hi, x.C, x.W, x.H, x.P, x.n, p.TW, p.TH, p.TN);
      maps.a[sidx][1] = passes >= 2 ? make_act_map(x.p.lo, x.C, x.W, x.H, x.P, x.n, p.TW, p.TH, p.TN) : maps.a[sidx][0];
    };
    xmaps(xk->x0, 2);
    if (xk->has_x1) xmaps(xk->x1, 3);
  }

  const double Mtot = (double)a0.n * a0.H * a0.W;
  const double flops = 2.0 * Mtot * (double)w.N * ((double)w.K + 64.0 * p.xkc);  // algorithmic (one product per MAC)
  // algorithmic bytes of one launch (DESIGN.md §4): every operand element read once in the formats the passes need, the
  // result written once in every format it is produced in
  const double a_bytes = Mtot * (Ctot + 64.0 * p.xkc) * 2.0 * (passes >= 2 ? 2 : 1);
  const double w_bytes = (double)w.N * (w.K + 64.0 * p.xkc) * 2.0 * (passes >= 3 ? 2 : 1);
  const double o_bytes = Mtot * nout * ((ep.out_f32 ? 4.0 : 0.0) + (ep.out_f16.hi ? 2.0 : 0.0) + (ep.out_f16.lo ? 2.0 : 0.0)) +
                         (ep.residual ? Mtot * nout * 4.0 : 0.0);
  const double bytes = a_bytes + w_bytes + o_bytes;  // per launch (a folded-upsample phase reads all of A and writes a quarter of the output)

  {
    // the folded-upsample conv runs its four output phases in ONE launch (grid.z = phase): weights are packed phase-major
    // [4][N][K], so one map over 4 N rows serves them all
    const __half* whi = w.p.hi;
    const __half* wlo = w.p.lo;
    const int wrows = (w.rows ? w.rows : w.N) * phases_out;
    const int bbox = pair ? BN / 2 : BN;
    maps.b[0] = make_w_map(whi, w.K, wrows, bbox, w.ld);
    maps.b[1] = maps.b[0];
    if (passes >= 3) maps.b[1] = make_w_map(wlo, w.K, wrows, bbox, w.ld);
    maps.bx[0] = maps.bx[1] = maps.b[0];
    if (xk) {
      const int xrows = xk->w.rows ? xk->w.rows : xk->w.N;
      maps.bx[0] = make_w_map(xk->w.p.hi, xk->w.K, xrows, bbox, xk->w.ld);
      maps.bx[1] = passes >= 3 ? make_w_map(xk->w.p.lo, xk->w.K, xrows, bbox, xk->w.ld) : maps.bx[0];
    }
    p.gn_slot0 = 0;
    p.up2 = 0, p.gn_phase_slots = (m_tiles / p.tiles_n) * split;
    if (kind == G_CONV3_UP2) {
      // output phase (a, b) in {0,1}^2 sees the 2x2 window of source pixels at rows {h-1+a, h+a}, columns {w-1+b, w+b}: the
      // kernel adds (a, b) = (blockIdx.z >> 1, blockIdx.z & 1) to the phase-0 taps and to the output pixel
      p.up2 = 1, p.oa = 0, p.ob = 0;
      for (int t = 0; t < 4; ++t) p.tap_dh[t] = (t >> 1) - 1, p.tap_dw[t] = (t & 1) - 1, p.tap_ph[t] = 0;
    }
    if (split > 1) {
      const size_t need = (size_t)split * (size_t)Mtot * w.N * sizeof(float);
      p.ws = reinterpret_cast<float*>(c.work.alloc(need));
      SDB_CHECK((long long)m_tiles * n_tiles * 2 <= 65536, "split-K ticket buffer");
      SDB_CHECK((long long)m_tiles * n_tiles * split <= 148, "split-K CTAs must be co-resident");
      p.tickets = c.splitk_tickets;
    }
    {
      // flops = algorithmic 2*M*N*K of this launch; issued = the tensor-core FLOPs the passes really execute
      static const bool dbg_on = getenv("SDB_GEMM_DBG") != nullptr;
      static long long* dbg_buf = nullptr;
      if (dbg_on) {
        if (!dbg_buf) SDB_CUDA(cudaMallocManaged(&dbg_buf, 16 * sizeof(long long)));
        SDB_CUDA(cudaStreamSynchronize(c.stream));
        memset(dbg_buf, 0, 16 * sizeof(long long));
        p.dbg = dbg_buf;
      }
      const std::string label = c.dbg_label;
      {
        KernelScope ks(c, KC_GEMM, flops * phases_out, bytes * phases_out, flops * passes * phases_out);
        gemm_tc_launch(maps, p, BN, passes, c.stream);
      }
      if (dbg_on) {  // bring-up aid: cycle stamps of CTA (0,0,0), printed relative to kernel entry
        SDB_CUDA(cudaStreamSynchronize(c.stream));
        fprintf(stderr, "gemm_dbg %s | cycles since entry: prologue %lld tma0 %lld landed %lld lastmma %lld accum %lld epi %lld exit %lld | chunk0: ld %lld stage %lld finish %lld (bias %lld loads0 %lld batch0 %lld)\n",
                label.c_str(), dbg_buf[1] - dbg_buf[0], dbg_buf[2] - dbg_buf[0], dbg_buf[3] - dbg_buf[0],
                dbg_buf[4] - dbg_buf[0], dbg_buf[5] - dbg_buf[0], dbg_buf[6] - dbg_buf[0], dbg_buf[7] - dbg_buf[0], dbg_buf[9] - dbg_buf[8], dbg_buf[10] - dbg_buf[9],
                dbg_buf[11] - dbg_buf[10], dbg_buf[12] - dbg_buf[10], dbg_buf[13] - dbg_buf[12], dbg_buf[14] - dbg_buf[13]);
      }
    }
    // (the split-K reduction happens inside the kernel: after a ticket rendezvous every split CTA folds its slice of the tile rows)
  }
}

}  // namespace sdb
