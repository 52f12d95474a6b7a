// runtime.cuh — context, arenas, weight registry, tensor-map construction, GEMM op builder.
#pragma once
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "common.cuh"
#include "attention.cuh"
#include "gemm_tc.cuh"
#include "kernels.cuh"

namespace sdb {

struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0, high = 0;
  void init(size_t bytes);
  void destroy();
  void* alloc(size_t bytes);
  template <class T>
  T* get(size_t count) {
    return reinterpret_cast<T*>(alloc(count * sizeof(T)));
  }
  void reset() { off = 0; }
};

enum TensorKind : int { K_CONV_W = 0, K_CONV_B, K_LIN_W, K_LIN_B, K_NORM_G, K_NORM_B, K_SCHED, K_EMB };
struct TensorInfo {
  std::string name;
  int64_t dims[4] = {1, 1, 1, 1};
  int ndim = 0;
  size_t offset = 0;  // float offset in the master arena
  int64_t count = 0;
  int kind = 0;       // TensorKind
  int fan_in = 1;
};

enum KernelClass : int {
  KC_GEMM = 0,
  KC_SPLITK,  // kept for the class table layout: the split-K fold now happens inside gemm_tc
  KC_ATTN,
  KC_GN_STATS,
  KC_PREP,
  KC_LAYERNORM,
  KC_SMALLCONV,
  KC_ELEMENTWISE,
  KC_COUNT
};

struct ProfEvent {
  int cls;
  cudaEvent_t a, b;
  double flops, bytes;
  std::string label;
};

// fp16 activation operand [n][P][H][W][C]
struct ActOp {
  Half2Ptr p;
  int n = 1, P = 1, H = 1, W = 1, C = 0;
};
// packed weight [N][K]
struct WeightOp {
  Half2Ptr p;
  int N = 0, K = 0;
  long long ld = 0;  // row stride in elements (0 -> K)
  int rows = 0;      // rows that really exist (0 -> N); rows in [rows, N) read as zero (TMA OOB fill)
};
// G_CONV3_S2: 3x3 stride 2 pad 1 (UNet downsample); G_CONV3_S2_PAD01: 3x3 stride 2 padded bottom/right only
// (the VAE encoder's PaddedConv2d(0,1,0,1), autoencoder/mod.rs:229-236). Both read a 4-phase-plane operand.
enum GemmKind : int { G_LINEAR = 0, G_CONV1 = 1, G_CONV3 = 2, G_CONV3_S2 = 3, G_CONV3_UP2 = 4, G_CONV3_S2_PAD01 = 5 };

// GroupNorm statistics a producer leaves beside its output tensor (gemm_tc.cuh: gn_part): [n][cap][C / bucket][2] floats.
// `slots` = partial slots really written per image (set by run_gemm; 0 = no statistics: the consumer computes its own).
struct GnPart {
  float* buf = nullptr;
  int cap = 0, bucket = 0, slots = 0;
};

struct Epilogue {
  // LayerNorm folded into the surrounding GEMMs (gemm_tc.cuh): producer side leaves row statistics of its output, consumer
  // side (weights carry gamma, `bias` carries beta^T W + b) normalises in its epilogue
  float* ln_out = nullptr;         // [rows][ln_slots(N)][2]
  const float* ln_in = nullptr;    // [rows][ln_in_slots][2]
  int ln_in_slots = 0, ln_C = 0;
  float ln_eps = 1e-5f;
  const float* ln_u_hi = nullptr;  // column sums of the hi halves of the folded weights (1- and 2-pass products)
  const float* ln_u_full = nullptr;  // column sums of hi + lo (3-pass products)
  Half2Ptr residual16;             // residual as an fp16 hi + lo pair (row stride ldc16) instead of `residual`
  GnPart* gn = nullptr;  // request statistics of the output (buf/cap/bucket preset by the caller)
  int gn_rpi = 0;        // G_LINEAR over tokens only: rows per image (G_CONV1 fills it from the operand geometry)
  float* out_f32 = nullptr;
  Half2Ptr out_f16;
  const float* bias = nullptr;
  const float* rowbias = nullptr;
  const float* residual = nullptr;
  int geglu = 0;
  int act = 0;    // 1 = QuickGELU
  int ldc = 0;    // 0 -> N (or N/2 for geglu)
  int ldc16 = 0;  // 0 -> N (or N/2 for geglu)
};

// a configuration scalar / small vector the reference's loaders read beside the tensors (dump-dir, dumpdir.cu):
// relpath (no ".npy") and the values it must hold for the compiled topology
struct MetaCheck {
  std::string relpath;
  std::vector<float> values;
  bool must_be_absent = false;  // e.g. a bias file on a bias-less Linear
};

struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::string err;
  Arena master, packed, work;
  std::vector<TensorInfo> tensors;
  std::unordered_map<std::string, int> index;
  bool finalized = false;
  std::vector<MetaCheck> meta;                       // dump-dir configuration files to validate
  std::unordered_set<std::string> group_norms;       // norm dirs that are GroupNorm (optional weight/bias on disk)
  std::unordered_map<std::string, float> norm_eps;   // per-norm eps read from a dump-dir (default 1e-5)
  // options
  int opt_precision = 0;  // 0 = per-layer policy, 1/2/3 = force
  int opt_graphs = 1;
  int opt_splitk = 1;
  int opt_pair_bn256 = 0;
  int opt_splitk_min_iters = 32, opt_splitk_chunk = 8;  // split-K: shortest K loop that is split, k-chunks kept per split
  int opt_skip_merge = 1; // ResBlock skip 1x1 conv folded into conv_out's K loop (needs raw16)
  int opt_raw16 = 1;      // epilogues also write the fp16 hi/lo copy a later raw-operand consumer needs (no staging launch)
  int opt_mlp_passes = 0;   // 0: the transformer MLP (GEGLU + ff) follows its level's pass policy; 1: single fp16 pass everywhere
  int opt_attn_split = 1;   // fused attention on the 3-pass levels takes q / k as fp16 hi + lo pairs (fp32-class logits)
  int opt_emb_hoist = 1;    // sample_latent computes the time-embedding rows of every timestep once per call (not once per step)
  int opt_prefetch_w = 0;   // 1: weight-bound GEMMs (<= 4 M tiles) prefetch their weight strip into L2 ahead of griddepcontrol.wait.
                            // Measured off (tools/step_time.py, same process): 143.38 ms per image with it, 142.59 ms without
  int opt_gn_epilogue = 1;  // GroupNorm statistics produced by the GEMM epilogue that writes the tensor (no stats pass, no rendezvous)
  int opt_cluster = 1;    // CTA pairs issue cta_group::2 MMAs (256 x BN) wherever the M-tile count is even and K is not split
  // profiling
  bool profiling = false;
  std::vector<ProfEvent> prof;
  int64_t launches = 0;
  double cls_ms[KC_COUNT] = {0}, cls_flops[KC_COUNT] = {0}, cls_bytes[KC_COUNT] = {0};
  double cls_issued[KC_COUNT] = {0};  // tensor-core FLOPs actually issued (x passes for split-fp16 products)
  int64_t cls_launches[KC_COUNT] = {0};
  // grow-only device staging for the host-buffer entry points (no cudaMalloc/cudaFree per call: each is a device-wide sync)
  struct IoBuf {
    void* p = nullptr;
    size_t cap = 0;
  } iobuf[8];
  void* io(int slot, size_t bytes);
  // grow-only device state of the samplers: slots 0-2 img2img (encoded image, noise, latent mask), which must survive the
  // work-arena reset between the encoder and the step loop; slot 3 the DPM-Solver++(2M) history x0_{i-1} and slot 4 the seeded
  // initial latent of sdb_sample_ex_dev, kept out of the work arena so that every sampler replays the same step graph. None is
  // ever one of the host wrappers' staging slots.
  IoBuf statebuf[8];
  void* state(int slot, size_t bytes);
  void io_destroy();  // frees iobuf and statebuf
  void* model = nullptr;  // Model* (model.cu)
  unsigned int* splitk_tickets = nullptr;  // 64K zeroed counters (gemm_tc split-K tile tickets)
  // SDB_DEBUG_SYNC=1: synchronise after every launch and report the failing op (bring-up aid)
  bool debug_sync = false;
  std::string dbg_label;

  float* master_ptr(const std::string& name);
  const TensorInfo& info(const std::string& name);
  bool has(const std::string& name) const { return index.count(name) != 0; }
};

struct KernelScope {  // RAII: counts a launch, optionally brackets it with events
  Ctx& c;
  int cls;
  bool on;
  ProfEvent ev;
  KernelScope(Ctx& c, int cls, double flops = 0, double bytes = 0, double issued = 0);
  ~KernelScope();
};
void profile_collect(Ctx& c);

// "extra K": operands read at the centre tap only, appended to a conv's K loop — the ResBlock's 1x1 skip conv
// (unet/mod.rs:729-731) folded into conv_out, so the block needs neither a separate launch nor a residual read
struct ExtraK {
  ActOp x0, x1;
  bool has_x1 = false;
  WeightOp w;  // [N][x0.C + x1.C]
};

// one tcgen05 GEMM / implicit conv (+ split-K reduction when chosen)
//   a0 (+a1 = channel concat), geometry kind, weights, passes (1..3), epilogue
void run_gemm(Ctx& c, int kind, const ActOp& a0, const ActOp* a1, const WeightOp& w, int passes, const Epilogue& ep,
              const ExtraK* xk = nullptr);

// fused attention over fp16 matrices:
//   q  [nb*q_rows][ldq]  head h at columns q_col0 + h*dpad (zero padded to dpad)
//   k  [nb*k_rows][ldk]  head h at columns k_col0 + h*dpad
//   vT [heads*d][ldv]    sample s at columns s*k_rows
//   out [nb*q_rows][ldo] head h at columns h*d
struct AttnOp {
  const __half* q = nullptr;
  int ldq = 0, q_col0 = 0, q_rows = 0;
  const __half* k = nullptr;
  int ldk = 0, k_col0 = 0, k_rows = 0;
  const __half* q_lo = nullptr;  // lo halves of q / k (same layout): both set -> the 3-term split QK^T (head dims 40 / 80)
  const __half* k_lo = nullptr;
  const __half* vT = nullptr;  // V^T [heads*d][ldv], or with v_mn = 1 the row-major V [nb*k_rows][ldv] (head-padded like k)
  int ldv = 0;
  int v_mn = 0, v_col0 = 0;
  int nb = 1, heads = 8, d = 0, dpad = 0, Nq = 0, Nk = 0;
  const int* kvlen = nullptr;
  int causal = 0;  // 1: key j visible to query i only if j <= i (CLIP, src/backend.rs:130-139)
  Half2Ptr out;
  int ldo = 0;
};
void run_attention(Ctx& c, const AttnOp& a);
// partial-sum slots per row that a LayerNorm-statistics producer of width N writes (N tiles of 160 x 2 chunk shares)
inline int ln_slots(int N) { return ((N + 159) / 160) * 2; }

const char* kernel_class_name(int cls);

}  // namespace sdb
