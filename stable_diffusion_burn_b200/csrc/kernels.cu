// kernels.cu — HBM-bound kernels around the tensor-core GEMMs: GroupNorm statistics, operand staging
// (GroupNorm-apply + SiLU + fp16 hi/lo split, upsample / stride-2 phase layouts), LayerNorm, the
// small CUDA-core convolutions (Cin = 4, Cout <= 4), sampler elementwise ops, weight packing.
// All activations are NHWC; loads/stores are 8- or 16-byte vectors, coalesced along channels.
#include "kernels.cuh"

#include <algorithm>

namespace sdb {

static inline int ceil_div(long long a, long long b) { return int((a + b - 1) / b); }

__device__ __forceinline__ void split_store8(const float (&f)[8], __half* hi, __half* lo) {
  __half2 h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = f2h2_sat(f[2 * j], f[2 * j + 1]);
  *reinterpret_cast<uint4*>(hi) = *reinterpret_cast<uint4*>(h);
  if (lo) {
    __half2 l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 hf = __half22float2(h[j]);
      l[j] = __floats2half2_rn(f[2 * j] - hf.x, f[2 * j + 1] - hf.y);
    }
    *reinterpret_cast<uint4*>(lo) = *reinterpret_cast<uint4*>(l);
  }
}

// ============================================================ GroupNorm statistics
// Deterministic two-level reduction (no floating-point atomics): every CTA reduces its pixel chunk per group in a
// fixed order and writes a partial; the last CTA of an image (ticket counter) folds the partials in chunk order.
__global__ void __launch_bounds__(256) gn_stats_kernel(const float* __restrict__ x0, int C0,
                                                       const float* __restrict__ x1, int C1, int HW, int pix_per_cta,
                                                       double* __restrict__ sums, float* __restrict__ partials,
                                                       unsigned int* __restrict__ tickets) {
  pdl_enter();
  __shared__ float s_pair[2][1280];  // per channel-pair (sum, sumsq), C <= 2560
  __shared__ bool s_last;
  const int n = blockIdx.y;
  const int C = C0 + C1, gs = C / 32;
  const int p0 = blockIdx.x * pix_per_cta;
  const int p1 = min(HW, p0 + pix_per_cta);
  // thread -> (channel pair, pixel lane): narrow tensors (C/2 < 256) spread the spare threads over pixels
  const int npair = C / 2;
  const int pg = npair >= 256 ? 1 : 256 / npair;          // pixel lanes per channel pair
  const int nslot = npair >= 256 ? npair : npair * pg;    // (pixel lane, pair) partials, <= 1280
  for (int slot = threadIdx.x; slot < nslot; slot += blockDim.x) {
    const int cp = slot % npair, pl = slot / npair;
    const int c = cp * 2;
    const float* ptr;
    int stride;
    if (c < C0) {
      ptr = x0 + (size_t)n * HW * C0 + c;
      stride = C0;
    } else {
      ptr = x1 + (size_t)n * HW * C1 + (c - C0);
      stride = C1;
    }
    float s = 0.f, q = 0.f;
    int p = p0 + pl;
    for (; p + 3 * pg < p1; p += 4 * pg) {
      float2 v0 = *reinterpret_cast<const float2*>(ptr + (size_t)p * stride);
      float2 v1 = *reinterpret_cast<const float2*>(ptr + (size_t)(p + pg) * stride);
      float2 v2 = *reinterpret_cast<const float2*>(ptr + (size_t)(p + 2 * pg) * stride);
      float2 v3 = *reinterpret_cast<const float2*>(ptr + (size_t)(p + 3 * pg) * stride);
      s += (v0.x + v0.y) + (v1.x + v1.y) + (v2.x + v2.y) + (v3.x + v3.y);
      q += (v0.x * v0.x + v0.y * v0.y) + (v1.x * v1.x + v1.y * v1.y) + (v2.x * v2.x + v2.y * v2.y) +
           (v3.x * v3.x + v3.y * v3.y);
    }
    for (; p < p1; p += pg) {
      float2 v = *reinterpret_cast<const float2*>(ptr + (size_t)p * stride);
      s += v.x + v.y;
      q += v.x * v.x + v.y * v.y;
    }
    s_pair[0][slot] = s;
    s_pair[1][slot] = q;
  }
  __syncthreads();
  const int chunks = gridDim.x;
  if (threadIdx.x < 64) {  // thread = (group, stat): fold the group's channel pairs in index order
    const int g = threadIdx.x >> 1, which = threadIdx.x & 1;
    const int pairs = gs / 2;
    float acc = 0.f;
    for (int l = 0; l < (npair >= 256 ? 1 : pg); ++l)
      for (int i = 0; i < pairs; ++i) acc += s_pair[which][l * npair + g * pairs + i];
    partials[((size_t)n * chunks + blockIdx.x) * 64 + threadIdx.x] = acc;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&tickets[n], 1u) == (unsigned)(chunks - 1);
  __syncthreads();
  if (s_last && threadIdx.x < 64) {
    __threadfence();
    double acc = 0.0;
    for (int ch = 0; ch < chunks; ++ch) acc += (double)partials[((size_t)n * chunks + ch) * 64 + threadIdx.x];
    sums[(size_t)n * 64 + threadIdx.x] = acc;  // [n][32][2]
  }
}

size_t gn_stats_partial_floats(int n, int HW) {
  int pix = (int)((((long long)HW * n) + 591) / 592);
  if (pix < 16) pix = 16;
  return (size_t)n * ceil_div(HW, pix) * 64;
}

void gn_stats_launch(const float* x0, int C0, const float* x1, int C1, int n, int HW, double* sums, float* partials,
                     unsigned int* tickets, cudaStream_t st) {
  SDB_CHECK((C0 + C1) % 64 == 0 && C0 % 2 == 0 && C0 + C1 <= 2560, "GroupNorm channels");
  int pix = (int)((((long long)HW * n) + 591) / 592);
  if (pix < 16) pix = 16;
  dim3 grid(ceil_div(HW, pix), n);
  launch_k(gn_stats_kernel, grid, dim3(256), 0, st, x0, C0, x1, C1, HW, pix, sums, partials, tickets);
  SDB_CUDA(cudaGetLastError());
}

// per-(image, channel) affine from the group sums: y = x*scale + shift
__device__ __forceinline__ void gn_affine(const double* sums, int n, int c, int gs, double inv_cnt, float eps,
                                          const float* gamma, const float* beta, float& scale, float& shift) {
  const int g = c / gs;
  const double s = sums[((size_t)n * 32 + g) * 2 + 0], q = sums[((size_t)n * 32 + g) * 2 + 1];
  const double mean = s * inv_cnt;
  double var = q * inv_cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  scale = rstd * gamma[c];
  shift = beta[c] - (float)mean * scale;
}

// ============================================================ operand staging
__global__ void __launch_bounds__(256)
prep_operand_kernel(const float* __restrict__ x0, int C0, const float* __restrict__ x1, int C1, int H, int W,
                    int pix_per_cta, int mode, const double* __restrict__ sums, const float* __restrict__ gamma,
                    const float* __restrict__ beta, float eps, __half* __restrict__ out_hi,
                    __half* __restrict__ out_lo) {
  pdl_enter();
  extern __shared__ float s_aff[];  // scale[C], shift[C]
  const int n = blockIdx.y;
  const int C = C0 + C1, HW = H * W;
  float* s_scale = s_aff;
  float* s_shift = s_aff + C;
  if (mode & PREP_NORM) {
    const int gs = C / 32;
    const double inv_cnt = 1.0 / ((double)gs * HW);
    for (int c = threadIdx.x; c < C; c += blockDim.x) gn_affine(sums, n, c, gs, inv_cnt, eps, gamma, beta, s_scale[c], s_shift[c]);
    __syncthreads();
  }
  const int p0 = blockIdx.x * pix_per_cta;
  const int p1 = min(HW, p0 + pix_per_cta);
  const int c8n = C / 8;
  const int items = (p1 - p0) * c8n;
  for (int i = threadIdx.x; i < items; i += blockDim.x) {
    const int p = p0 + i / c8n;
    const int c = (i % c8n) * 8;
    const float* src = (c < C0) ? x0 + ((size_t)n * HW + p) * C0 + c : x1 + ((size_t)n * HW + p) * C1 + (c - C0);
    float4 a = *reinterpret_cast<const float4*>(src);
    float4 b = *reinterpret_cast<const float4*>(src + 4);
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    if (mode & PREP_NORM) {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = f[j] * s_scale[c + j] + s_shift[c + j];
    }
    if (mode & PREP_SILU) {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j]);
    }
    const int h = p / W, w = p % W;
    if (mode & PREP_UP2) {
      const size_t base = (((size_t)n * 2 * H + 2 * h) * 2 * W + 2 * w) * C + c;
      const size_t rowstride = (size_t)2 * W * C;
      split_store8(f, out_hi + base, out_lo ? out_lo + base : nullptr);
      split_store8(f, out_hi + base + C, out_lo ? out_lo + base + C : nullptr);
      split_store8(f, out_hi + base + rowstride, out_lo ? out_lo + base + rowstride : nullptr);
      split_store8(f, out_hi + base + rowstride + C, out_lo ? out_lo + base + rowstride + C : nullptr);
    } else if (mode & PREP_PHASE2) {
      const int ph = (h & 1) * 2 + (w & 1);
      const size_t o = ((((size_t)n * 4 + ph) * (H / 2) + (h >> 1)) * (W / 2) + (w >> 1)) * C + c;
      split_store8(f, out_hi + o, out_lo ? out_lo + o : nullptr);
    } else {
      const size_t o = ((size_t)n * HW + p) * C + c;
      split_store8(f, out_hi + o, out_lo ? out_lo + o : nullptr);
    }
  }
}

void prep_operand_launch(const float* x0, int C0, const float* x1, int C1, int n, int H, int W, int mode,
                         const double* sums, const float* gamma, const float* beta, float eps, Half2Ptr out,
                         cudaStream_t st) {
  const int C = C0 + C1, HW = H * W;
  SDB_CHECK(C % 8 == 0 && C0 % 8 == 0, "operand channels must be multiples of 8");
  int pix = (int)((((long long)HW * n) + 1183) / 1184);
  if (pix < 8) pix = 8;
  dim3 grid(ceil_div(HW, pix), n);
  const size_t smem = (mode & PREP_NORM) ? (size_t)2 * C * sizeof(float) : 0;
  launch_k(prep_operand_kernel, grid, dim3(256), smem, st, x0, C0, x1, C1, H, W, pix, mode, sums, gamma, beta, eps, out.hi, out.lo);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ fused GroupNorm: statistics + apply in ONE launch
// Phase 1: per-CTA group partials of the CTA's pixel chunk (fixed-order, deterministic), published to global memory.
// After an in-kernel rendezvous of the image's CTAs every CTA folds all partials (same order everywhere). Phase 2:
// normalise + SiLU + fp16 hi/lo split of the same chunk (second read hits L2). The grid never exceeds 4 CTAs per SM,
// so every CTA is resident and the wait cannot deadlock.
__global__ void __launch_bounds__(256)
gn_fused_kernel(const float* __restrict__ x0, int C0, const float* __restrict__ x1, int C1, int H, int W, int pix_per_cta,
                int silu, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                __half* __restrict__ out_hi, __half* __restrict__ out_lo, float* __restrict__ partials,
                unsigned int* __restrict__ tickets) {
  pdl_enter();
  extern __shared__ float s_dyn[];  // scale[C], shift[C]
  __shared__ float s_pair[2][1280];
  const int n = blockIdx.y;
  const int C = C0 + C1, gs = C / 32, HW = H * W;
  const int p0 = blockIdx.x * pix_per_cta;
  const int p1 = min(HW, p0 + pix_per_cta);
  // ---- phase 1
  // thread -> (channel pair, pixel lane): narrow tensors (C/2 < 256) spread the spare threads over pixels
  const int npair = C / 2;
  const int pg = npair >= 256 ? 1 : 256 / npair;          // pixel lanes per channel pair
  const int nslot = npair >= 256 ? npair : npair * pg;    // (pixel lane, pair) partials, <= 1280
  for (int slot = threadIdx.x; slot < nslot; slot += blockDim.x) {
    const int cp = slot % npair, pl = slot / npair;
    const int c = cp * 2;
    const float* ptr;
    int stride;
    if (c < C0) {
      ptr = x0 + (size_t)n * HW * C0 + c;
      stride = C0;
    } else {
      ptr = x1 + (size_t)n * HW * C1 + (c - C0);
      stride = C1;
    }
    float s = 0.f, q = 0.f;
    int p = p0 + pl;
    for (; p + 3 * pg < p1; p += 4 * pg) {
      float2 v0 = *reinterpret_cast<const float2*>(ptr + (size_t)p * stride);
      float2 v1 = *reinterpret_cast<const float2*>(ptr + (size_t)(p + pg) * stride);
      float2 v2 = *reinterpret_cast<const float2*>(ptr + (size_t)(p + 2 * pg) * stride);
      float2 v3 = *reinterpret_cast<const float2*>(ptr + (size_t)(p + 3 * pg) * stride);
      s += (v0.x + v0.y) + (v1.x + v1.y) + (v2.x + v2.y) + (v3.x + v3.y);
      q += (v0.x * v0.x + v0.y * v0.y) + (v1.x * v1.x + v1.y * v1.y) + (v2.x * v2.x + v2.y * v2.y) +
           (v3.x * v3.x + v3.y * v3.y);
    }
    for (; p < p1; p += pg) {
      float2 v = *reinterpret_cast<const float2*>(ptr + (size_t)p * stride);
      s += v.x + v.y;
      q += v.x * v.x + v.y * v.y;
    }
    s_pair[0][slot] = s;
    s_pair[1][slot] = q;
  }
  __syncthreads();
  const int chunks = gridDim.x;
  if (threadIdx.x < 64) {
    const int g = threadIdx.x >> 1, which = threadIdx.x & 1;
    const int pairs = gs / 2;
    float acc = 0.f;
    for (int l = 0; l < (npair >= 256 ? 1 : pg); ++l)
      for (int i = 0; i < pairs; ++i) acc += s_pair[which][l * npair + g * pairs + i];
    partials[((size_t)n * chunks + blockIdx.x) * 64 + threadIdx.x] = acc;
  }
  __threadfence();
  __syncthreads();
  // ---- rendezvous of the image's CTAs (all co-resident), then EVERY CTA folds the partials itself in the same fixed
  // order: no single-CTA serial tail and no second flag round trip; the result is identical in every CTA.
  if (threadIdx.x == 0) {
    atomicAdd(&tickets[n], 1u);
    const long long t0 = clock64();
    while (atomicAdd(&tickets[n], 0u) < (unsigned)chunks) {
      __nanosleep(64);
      if (clock64() - t0 > 4000000000ll) __trap();  // ~2 s: a lost CTA becomes a launch failure, not a hung GPU
    }
    __threadfence();
  }
  __syncthreads();
  __shared__ double s_fold[4][64];
  __shared__ double s_sum[64];
  {
    const int stat = threadIdx.x & 63, part = threadIdx.x >> 6;
    const int per = (chunks + 3) / 4;
    const int c0 = part * per, c1 = min(chunks, c0 + per);
    const float* src = partials + (size_t)n * chunks * 64 + stat;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int ch = c0;
    for (; ch + 3 < c1; ch += 4) {
      const float v0 = __ldcg(src + (size_t)ch * 64), v1 = __ldcg(src + (size_t)(ch + 1) * 64);
      const float v2 = __ldcg(src + (size_t)(ch + 2) * 64), v3 = __ldcg(src + (size_t)(ch + 3) * 64);
      a0 += (double)v0, a1 += (double)v1, a2 += (double)v2, a3 += (double)v3;
    }
    for (; ch < c1; ++ch) a0 += (double)__ldcg(src + (size_t)ch * 64);
    s_fold[part][stat] = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();
  if (threadIdx.x < 64)
    s_sum[threadIdx.x] = ((s_fold[0][threadIdx.x] + s_fold[1][threadIdx.x]) + s_fold[2][threadIdx.x]) + s_fold[3][threadIdx.x];
  __syncthreads();
  // ---- phase 2
  float* s_scale = s_dyn;
  float* s_shift = s_dyn + C;
  {
    const double inv_cnt = 1.0 / ((double)gs * HW);
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      const int g = c / gs;
      const double sm = s_sum[g * 2 + 0], sq = s_sum[g * 2 + 1];
      const double mean = sm * inv_cnt;
      double var = sq * inv_cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      const float rstd = (float)(1.0 / sqrt(var + (double)eps));
      const float sc = rstd * gamma[c];
      s_scale[c] = sc;
      s_shift[c] = beta[c] - (float)mean * sc;
    }
  }
  __syncthreads();
  const int c8n = C / 8;
  const int items = (p1 - p0) * c8n;
  for (int i = threadIdx.x; i < items; i += blockDim.x) {
    const int p = p0 + i / c8n;
    const int c = (i % c8n) * 8;
    const float* src = (c < C0) ? x0 + ((size_t)n * HW + p) * C0 + c : x1 + ((size_t)n * HW + p) * C1 + (c - C0);
    float4 a = *reinterpret_cast<const float4*>(src);
    float4 b = *reinterpret_cast<const float4*>(src + 4);
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = f[j] * s_scale[c + j] + s_shift[c + j];
    if (silu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j]);
    }
    const size_t o = ((size_t)n * HW + p) * C + c;
    split_store8(f, out_hi + o, out_lo ? out_lo + o : nullptr);
  }
}

// ============================================================ GroupNorm apply from producer-side statistics
// The GEMM that wrote the tensor also left per-(image, slot, channel-bucket) partial sums (gemm_tc.cuh: gn_part). Every CTA folds
// the partials of its image in a fixed order (fp64), derives the per-channel affine and makes ONE pass over its pixel chunk:
// x read once, no statistics pass, no grid rendezvous. Reads the two sources of cat([x0, x1]) directly.
__global__ void __launch_bounds__(256)
gn_apply_kernel(const GnSrc s0, const GnSrc s1, int bucket, int H, int W, int pix_per_cta, int silu,
                const float* __restrict__ gamma, const float* __restrict__ beta, float eps, __half* __restrict__ out_hi,
                __half* __restrict__ out_lo) {
  pdl_enter();
  extern __shared__ float s_dyn[];  // scale[C], shift[C]
  __shared__ double s_bsum[2 * 256];  // (sum, sumsq) per channel bucket of the concat, C / bucket <= 256
  __shared__ double s_gsum[64];
  const int n = blockIdx.y;
  const int C0 = s0.C, C1 = s1.C, C = C0 + C1, gs = C / 32, HW = H * W;
  const int nb0 = C0 / bucket, nbt = C / bucket;
  // fold of the producer's partial slots. A serial walk would be a chain of L2 round trips (~0.35 us each): the slots of one
  // (bucket, stat) item are spread over `lanes` threads, four loads in flight each, and the lanes are combined in index order
  // (fixed order everywhere -> every CTA of the image derives bit-identical statistics)
  __shared__ double s_lane[512];
  {
    const int items = 2 * nbt;
    const int lanes = items >= 256 ? 1 : 256 / items;
    for (int idx = threadIdx.x; idx < items * lanes; idx += blockDim.x) {
      const int t = idx % items, lane = idx / items;
      const int b = t >> 1, which = t & 1;
      const GnSrc& s = b < nb0 ? s0 : s1;
      const int nbk = s.C / bucket, bb = b < nb0 ? b : b - nb0;
      const float* p = s.part + ((size_t)n * s.cap * nbk + bb) * 2 + which;
      const size_t st = (size_t)nbk * 2;
      double a = 0.0;
      int sl = lane;
      for (; sl + 3 * lanes < s.slots; sl += 4 * lanes) {
        const float v0 = __ldcg(p + sl * st), v1 = __ldcg(p + (sl + lanes) * st);
        const float v2 = __ldcg(p + (sl + 2 * lanes) * st), v3 = __ldcg(p + (sl + 3 * lanes) * st);
        a += (double)v0, a += (double)v1, a += (double)v2, a += (double)v3;
      }
      for (; sl < s.slots; sl += lanes) a += (double)__ldcg(p + sl * st);
      s_lane[lane * items + t] = a;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < items; t += blockDim.x) {
      double a = 0.0;
      for (int l = 0; l < lanes; ++l) a += s_lane[l * items + t];
      s_bsum[t] = a;
    }
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int g = threadIdx.x >> 1, which = threadIdx.x & 1, bpg = gs / bucket;
    double a = 0.0;
    for (int i = 0; i < bpg; ++i) a += s_bsum[(g * bpg + i) * 2 + which];
    s_gsum[threadIdx.x] = a;
  }
  __syncthreads();
  float* s_scale = s_dyn;
  float* s_shift = s_dyn + C;
  {
    const double inv_cnt = 1.0 / ((double)gs * HW);
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      const int g = c / gs;
      const double mean = s_gsum[g * 2] * inv_cnt;
      double var = s_gsum[g * 2 + 1] * inv_cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      const float sc = (float)(1.0 / sqrt(var + (double)eps)) * gamma[c];
      s_scale[c] = sc;
      s_shift[c] = beta[c] - (float)mean * sc;
    }
  }
  __syncthreads();
  const int p0 = blockIdx.x * pix_per_cta, p1 = min(HW, p0 + pix_per_cta);
  const int c8n = C / 8;
  const int items = (p1 - p0) * c8n;
  const float* x0 = s0.x;
  const float* x1 = s1.x;
  auto src_of = [&](int i, int& p, int& c) {
    p = p0 + i / c8n;
    c = (i - (i / c8n) * c8n) * 8;
    return (c < C0) ? x0 + ((size_t)n * HW + p) * C0 + c : x1 + ((size_t)n * HW + p) * C1 + (c - C0);
  };
  auto finish = [&](float4 a, float4 b, int p, int c) {
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], s_scale[c + j], s_shift[c + j]);
    if (silu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j]);
    }
    const size_t o = ((size_t)n * HW + p) * C + c;
    split_store8(f, out_hi + o, out_lo ? out_lo + o : nullptr);
  };
  // two items per thread and iteration: 4 independent 16-byte loads in flight before the first use
  int i = threadIdx.x;
  for (; i + (int)blockDim.x < items; i += 2 * blockDim.x) {
    int pa, ca, pb, cb;
    const float* sa = src_of(i, pa, ca);
    const float* sb = src_of(i + blockDim.x, pb, cb);
    const float4 a0 = __ldcs(reinterpret_cast<const float4*>(sa)), a1 = __ldcs(reinterpret_cast<const float4*>(sa + 4));
    const float4 b0 = __ldcs(reinterpret_cast<const float4*>(sb)), b1 = __ldcs(reinterpret_cast<const float4*>(sb + 4));
    finish(a0, a1, pa, ca);
    finish(b0, b1, pb, cb);
  }
  if (i < items) {
    int pa, ca;
    const float* sa = src_of(i, pa, ca);
    finish(*reinterpret_cast<const float4*>(sa), *reinterpret_cast<const float4*>(sa + 4), pa, ca);
  }
}

// Large images leave thousands of partial slots (one per 128-pixel tile): a first pass folds groups of 64 slots (fp64 inside,
// fixed order) so that the apply kernel's per-CTA fold stays short. in [n][cap][nbk][2] -> out [n][ceil(slots/64)][nbk][2].
__global__ void __launch_bounds__(256)
gn_fold_kernel(const float* __restrict__ part, int cap, int slots, int nbk2, float* __restrict__ out) {
  pdl_enter();
  const int n = blockIdx.y, chunk = blockIdx.x, nchunks = gridDim.x;
  const int s0 = chunk * 64, s1 = min(slots, s0 + 64);
  for (int t = threadIdx.x; t < nbk2; t += blockDim.x) {
    const float* p = part + ((size_t)n * cap + s0) * nbk2 + t;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int sl = 0;
    const int cnt = s1 - s0;
    for (; sl + 3 < cnt; sl += 4) {
      a0 += (double)__ldcg(p + (size_t)sl * nbk2), a1 += (double)__ldcg(p + (size_t)(sl + 1) * nbk2);
      a2 += (double)__ldcg(p + (size_t)(sl + 2) * nbk2), a3 += (double)__ldcg(p + (size_t)(sl + 3) * nbk2);
    }
    for (; sl < cnt; ++sl) a0 += (double)__ldcg(p + (size_t)sl * nbk2);
    out[((size_t)n * nchunks + chunk) * nbk2 + t] = (float)((a0 + a1) + (a2 + a3));
  }
}
int gn_fold_slots(int slots) { return (slots + 63) / 64; }
void gn_fold_launch(const float* part, int cap, int slots, int nbk, int n, float* out, cudaStream_t st) {
  dim3 grid(gn_fold_slots(slots), n);
  launch_k(gn_fold_kernel, grid, dim3(256), 0, st, part, cap, slots, nbk * 2, out);
  SDB_CUDA(cudaGetLastError());
}

// group sums [n][32][2] (double) of ONE tensor from the producer's (possibly pre-folded) partial slots: what gn_stats_kernel
// computes by reading the tensor, here from a few KB of partials
__global__ void __launch_bounds__(256)
gn_sums_from_partials_kernel(const float* __restrict__ part, int cap, int slots, int nbk, int bpg, double* __restrict__ sums) {
  pdl_enter();
  __shared__ double s_b[512];
  const int n = blockIdx.x;
  for (int t = threadIdx.x; t < 2 * nbk; t += blockDim.x) {
    const float* p = part + (size_t)n * cap * nbk * 2 + t;
    double a = 0.0;
    for (int sl = 0; sl < slots; ++sl) a += (double)__ldcg(p + (size_t)sl * nbk * 2);
    s_b[t] = a;
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int g = threadIdx.x >> 1, which = threadIdx.x & 1;
    double a = 0.0;
    for (int i = 0; i < bpg; ++i) a += s_b[(g * bpg + i) * 2 + which];
    sums[(size_t)n * 64 + threadIdx.x] = a;
  }
}
void gn_sums_from_partials_launch(const float* part, int cap, int slots, int nbk, int C, int bucket, int n, double* sums,
                                  cudaStream_t st) {
  SDB_CHECK(nbk <= 256 && (C / 32) % bucket == 0, "group sums from partials: geometry");
  launch_k(gn_sums_from_partials_kernel, dim3(n), dim3(256), 0, st, part, cap, slots, nbk, (C / 32) / bucket, sums);
  SDB_CUDA(cudaGetLastError());
}

int g_gn_apply_ctas = 592;  // measured (tools/step_time.py, ms per image): 1184 ?, 592 146.1, 296 149.3, 148 155.5
void gn_apply_launch(const GnSrc& s0, const GnSrc& s1, int bucket, int n, int H, int W, int silu, const float* gamma,
                     const float* beta, float eps, Half2Ptr out, cudaStream_t st) {
  const int C = s0.C + s1.C, HW = H * W;
  SDB_CHECK(C % 64 == 0 && s0.C % 8 == 0 && C <= 2560 && bucket > 0 && s0.C % bucket == 0 && s1.C % bucket == 0 &&
                (C / 32) % bucket == 0 && C / bucket <= 256,
            "GroupNorm apply: channel / bucket geometry");
  // no co-residency constraint any more; every CTA repeats the fold of its image's partials (8-24 KB from L2), so the grid is
  // kept to g_gn_apply_ctas CTAs (4 per SM by default), at least one pixel each
  int pix = (int)((((long long)HW * n) + g_gn_apply_ctas - 1) / g_gn_apply_ctas);
  if (pix < 1) pix = 1;
  dim3 grid(ceil_div(HW, pix), n);
  launch_k(gn_apply_kernel, grid, dim3(256), (size_t)2 * C * sizeof(float), st, s0, s1, bucket, H, W, pix, silu, gamma, beta, eps,
           out.hi, out.lo);
  SDB_CUDA(cudaGetLastError());
}

int g_gn_min_pix = 1;  // pixels per CTA floor: small feature maps are latency-bound, so they get many small CTAs
static int gn_fused_pix(int n, int HW) {
  int pix = (int)((((long long)HW * n) + 295) / 296);  // <= 296 CTAs (2 per SM): short fold, always co-resident
  return pix < g_gn_min_pix ? g_gn_min_pix : pix;
}
size_t gn_fused_partial_floats(int n, int HW) { return (size_t)n * ceil_div(HW, gn_fused_pix(n, HW)) * 64; }

void gn_fused_launch(const float* x0, int C0, const float* x1, int C1, int n, int H, int W, int silu, const float* gamma,
                     const float* beta, float eps, Half2Ptr out, float* partials, unsigned int* tickets, cudaStream_t st) {
  const int C = C0 + C1, HW = H * W;
  SDB_CHECK(C % 64 == 0 && C0 % 8 == 0 && C <= 2560, "GroupNorm channels");
  const int pix = gn_fused_pix(n, HW);
  dim3 grid(ceil_div(HW, pix), n);
  SDB_CHECK((long long)grid.x * grid.y <= 592, "fused GroupNorm grid must stay co-resident");
  launch_k(gn_fused_kernel, grid, dim3(256), (size_t)2 * C * sizeof(float), st, x0, C0, x1, C1, H, W, pix, silu, gamma, beta, eps, out.hi,
           out.lo, partials, tickets);
  SDB_CUDA(cudaGetLastError());
}

__global__ void __launch_bounds__(256)
gn_apply_f32_kernel(const float* __restrict__ x, int C, int HW, int silu, const double* __restrict__ sums,
                    const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float* __restrict__ y) {
  const int n = blockIdx.y;
  const int gs = C / 32;
  const double inv_cnt = 1.0 / ((double)gs * HW);
  const size_t total = (size_t)HW * C;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    float sc, sh;
    gn_affine(sums, n, c, gs, inv_cnt, eps, gamma, beta, sc, sh);
    float v = x[(size_t)n * total + i] * sc + sh;
    y[(size_t)n * total + i] = silu ? silu_f(v) : v;
  }
}
void gn_apply_f32_launch(const float* x, int C, int n, int HW, int silu, const double* sums, const float* gamma,
                         const float* beta, float eps, float* y, cudaStream_t st) {
  dim3 grid(ceil_div((long long)HW * C, 256 * 8), n);
  gn_apply_f32_kernel<<<grid, 256, 0, st>>>(x, C, HW, silu, sums, gamma, beta, eps, y);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ LayerNorm: one warp per row
template <int MAXV>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* __restrict__ x, int rows, int C, const float* __restrict__ gamma,
                 const float* __restrict__ beta, float eps, __half* __restrict__ out_hi, __half* __restrict__ out_lo,
                 float* __restrict__ out_f32) {
  pdl_enter();
  const int row = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int c8n = C / 8;
  const float* xr = x + (size_t)row * C;
  float v[MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int c8 = lane + k * 32;
    if (c8 < c8n) {
      float4 a = *reinterpret_cast<const float4*>(xr + c8 * 8);
      float4 b = *reinterpret_cast<const float4*>(xr + c8 * 8 + 4);
      v[k][0] = a.x, v[k][1] = a.y, v[k][2] = a.z, v[k][3] = a.w, v[k][4] = b.x, v[k][5] = b.y, v[k][6] = b.z, v[k][7] = b.w;
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[k][j];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)C;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int c8 = lane + k * 32;
    if (c8 < c8n) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[k][j] - mean;
        q += d * d;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / (float)C + eps);
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int c8 = lane + k * 32;
    if (c8 < c8n) {
      float f[8];
      const int c = c8 * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = (v[k][j] - mean) * rstd * gamma[c + j] + beta[c + j];
      if (out_hi) split_store8(f, out_hi + (size_t)row * C + c, out_lo ? out_lo + (size_t)row * C + c : nullptr);
      if (out_f32) {
        *reinterpret_cast<float4*>(out_f32 + (size_t)row * C + c) = make_float4(f[0], f[1], f[2], f[3]);
        *reinterpret_cast<float4*>(out_f32 + (size_t)row * C + c + 4) = make_float4(f[4], f[5], f[6], f[7]);
      }
    }
  }
}
void layernorm_launch(const float* x, int rows, int C, const float* gamma, const float* beta, float eps,
                      Half2Ptr out, float* out_f32, cudaStream_t st) {
  SDB_CHECK(C % 8 == 0 && C <= 1280, "LayerNorm width");
  const int grid = ceil_div(rows, 8);
  if (C <= 512)
    launch_k(layernorm_kernel<2>, dim3(grid), dim3(256), 0, st, x, rows, C, gamma, beta, eps, out.hi, out.lo, out_f32);
  else
    launch_k(layernorm_kernel<5>, dim3(grid), dim3(256), 0, st, x, rows, C, gamma, beta, eps, out.hi, out.lo, out_f32);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ conversions
__global__ void convert_f16_kernel(const float* __restrict__ x, long long count8, __half* __restrict__ hi,
                                   __half* __restrict__ lo) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count8; i += (long long)gridDim.x * blockDim.x) {
    float4 a = *reinterpret_cast<const float4*>(x + i * 8);
    float4 b = *reinterpret_cast<const float4*>(x + i * 8 + 4);
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    split_store8(f, hi + i * 8, lo ? lo + i * 8 : nullptr);
  }
}
void convert_f16_launch(const float* x, long long count, Half2Ptr out, cudaStream_t st) {
  SDB_CHECK(count % 8 == 0, "convert count");
  const long long c8 = count / 8;
  int grid = (int)((c8 + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  convert_f16_kernel<<<grid, 256, 0, st>>>(x, c8, out.hi, out.lo);
  SDB_CUDA(cudaGetLastError());
}

__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, int C, int HW, float* __restrict__ y, long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    const long long r = i / C;
    const int p = int(r % HW);
    const long long n = r / HW;
    y[i] = x[(n * C + c) * HW + p];
  }
}
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ x, int C, int HW, float* __restrict__ y, long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = int(i % HW);
    const long long r = i / HW;
    const int c = int(r % C);
    const long long n = r / C;
    y[i] = x[(n * HW + p) * C + c];
  }
}
void nchw_to_nhwc_launch(const float* x, int n, int C, int H, int W, float* y, cudaStream_t st) {
  const long long total = (long long)n * C * H * W;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  nchw_to_nhwc_kernel<<<grid, 256, 0, st>>>(x, C, H * W, y, total);
  SDB_CUDA(cudaGetLastError());
}
void nhwc_to_nchw_launch(const float* x, int n, int C, int H, int W, float* y, cudaStream_t st) {
  const long long total = (long long)n * C * H * W;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  nhwc_to_nchw_kernel<<<grid, 256, 0, st>>>(x, C, H * W, y, total);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ conv 3x3, Cin = 4 (fp32, CUDA cores)
// block = 64 pixels x (Cout/..) ; thread (pix, co-lane): weights staged in smem as [36][Cout]
__global__ void __launch_bounds__(256)
conv3x3_cin4_kernel(const float* __restrict__ x, int H, int W, const float* __restrict__ w, const float* __restrict__ b,
                    int Cout, const float* __restrict__ pre_w, const float* __restrict__ pre_b, float pre_scale,
                    float* __restrict__ y, __half* __restrict__ y_hi, __half* __restrict__ y_lo) {
  pdl_enter();
  extern __shared__ float sm[];
  float* s_w = sm;                  // [36][Cout]
  float* s_in = sm + 36 * Cout;     // [PIX][36]
  constexpr int PIX = 32;
  const int n = blockIdx.y;
  const int HW = H * W;
  const int p0 = blockIdx.x * PIX;
  for (int i = threadIdx.x; i < 36 * Cout; i += blockDim.x) {
    const int k = i / Cout, co = i % Cout;  // k = ci*9 + tap (OIHW inner order)
    s_w[i] = w[(size_t)co * 36 + k];
  }
  for (int i = threadIdx.x; i < PIX * 36; i += blockDim.x) {
    const int pl = i / 36, k = i % 36;
    const int ci = k / 9, tap = k % 9;
    const int p = p0 + pl;
    float v = 0.f;
    if (p < HW) {
      const int h = p / W + tap / 3 - 1, ww = p % W + tap % 3 - 1;
      if (h >= 0 && h < H && ww >= 0 && ww < W) {
        const float* xp = x + (size_t)n * 4 * HW + (size_t)h * W + ww;
        if (pre_w) {
          float acc = pre_b[ci];
#pragma unroll
          for (int cj = 0; cj < 4; ++cj) acc += pre_w[ci * 4 + cj] * (xp[(size_t)cj * HW] * pre_scale);
          v = acc;
        } else {
          v = xp[(size_t)ci * HW];
        }
      }
    }
    s_in[i] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < PIX * Cout; i += blockDim.x) {
    const int pl = i / Cout, co = i % Cout;
    const int p = p0 + pl;
    if (p >= HW) continue;
    float acc = b ? b[co] : 0.f;
#pragma unroll
    for (int k = 0; k < 36; ++k) acc += s_in[pl * 36 + k] * s_w[k * Cout + co];
    const size_t o = ((size_t)n * HW + p) * Cout + co;
    y[o] = acc;
    if (y_hi) {  // fp16 hi/lo copy for a consumer that takes this tensor as a raw GEMM operand
      const __half h = __float2half_rn(acc);
      y_hi[o] = h;
      if (y_lo) y_lo[o] = __float2half_rn(acc - __half2float(h));
    }
  }
}
void conv3x3_cin4_launch(const float* x_nchw, int n, int H, int W, const float* w, const float* b, int Cout,
                         const float* pre_w, const float* pre_b, float pre_scale, float* y, Half2Ptr y16, cudaStream_t st) {
  const size_t smem = (size_t)(36 * Cout + 32 * 36) * sizeof(float);
  static DeviceOnce once;
  if (once.first())
    SDB_CUDA(cudaFuncSetAttribute(conv3x3_cin4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  dim3 grid(ceil_div(H * W, 32), n);
  launch_k(conv3x3_cin4_kernel, grid, dim3(256), smem, st, x_nchw, H, W, w, b, Cout, pre_w, pre_b, pre_scale, y, y16.hi,
           y16.lo);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ conv 3x3, Cout <= 8, fused GroupNorm + SiLU (fp32, CUDA cores)
// The last conv of the UNet (320 -> 4), of the VAE decoder (128 -> 3 at 512x512: 134 MB of input) and of the encoder (512 -> 8).
// HBM-bound by construction (Cout is tiny), so the kernel is organised around reading x ONCE with wide coalesced loads:
//   CTA = 8 x 32 output pixels, 256 threads, one pixel each; channels in chunks of 16. Per chunk the (8+2) x (32+2) halo tile is
//   loaded (float4, 64 B contiguous per pixel), GroupNorm + SiLU applied on the way in, and stored channel-quad-major
//   [4][pixel][4] so that the warp's float4 reads are conflict-free; the chunk's weights sit beside it (broadcast reads).
// Each x element crosses HBM/L2 1.33 times (halo), against 9 times for the tap-by-tap warp-per-pixel kernel this replaces
// (512 us -> ~70 us on the VAE's last conv).
// TH = rows of the CTA tile (threads = 32 * TH): 8 for large images; 2 for small ones, where an 8-row tile would leave most SMs
// idle (UNet conv_out at 64x64, batch 2: 32 CTAs with TH = 8 -> 140 us). With so few warps per SM nothing hides the latency of a
// chunk's loads, so the small variant takes 64 channels per round (5 rounds for 320 channels instead of 20).
// KS = channel-split groups inside the CTA (threads = 32 * TH * KS): group ks takes the channel chunks ks, ks + KS, ... with its own
// halo tile and weight slice, and the groups' partial sums are added in group order at the end (deterministic). The small-image
// variant uses it to put 10 warps on an SM instead of 2: at 64x64, batch 2 the 128 two-warp CTAs left every SM with two warps
// and the kernel latency-bound at 136 us (ncu launch list, profiles/r2_launches_summary.md).
template <int COUT, int TH, int CK, int KS = 1>
__global__ void __launch_bounds__(32 * TH * KS)
conv3x3_small_cout_kernel(const float* __restrict__ x, int H, int W, int C, const double* __restrict__ sums,
                          const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                          const float* __restrict__ wp, const float* __restrict__ b, float* __restrict__ y) {
  pdl_enter();
  constexpr int TW = 32, HP = TH + 2, WP = TW + 2, NPIX = HP * WP, GT = 32 * TH;  // GT = threads of one group
  constexpr int GROUP_F4 = (CK / 4) * NPIX + 9 * COUT * (CK / 4);                  // float4s of one group's tile + weights
  extern __shared__ float sm[];
  float* s_scale = sm;                           // [C]
  float* s_shift = sm + C;                       // [C]
  const int ks = threadIdx.x / GT, gtid = threadIdx.x - ks * GT;
  float4* s_act = reinterpret_cast<float4*>(sm + 2 * C) + (size_t)ks * GROUP_F4;   // [CK/4][NPIX] float4 (this group's)
  float4* s_w = s_act + (CK / 4) * NPIX;         // [9][COUT][CK/4] float4
  const int n = blockIdx.z;
  const int HW = H * W;
  const int h0 = blockIdx.y * TH, w0 = blockIdx.x * TW;
  {
    const int gs = C / 32;
    const double inv_cnt = 1.0 / ((double)gs * HW);
    for (int c = threadIdx.x; c < C; c += blockDim.x) gn_affine(sums, n, c, gs, inv_cnt, eps, gamma, beta, s_scale[c], s_shift[c]);
  }
  const int tx = gtid & 31, ty = gtid >> 5;
  float acc[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) acc[o] = 0.f;
  for (int c0 = ks * CK; c0 < C; c0 += CK * KS) {  // the launcher guarantees (C / CK) % KS == 0: every group runs the same rounds
    __syncthreads();  // the previous chunk's reads are done (and, first time round, the affine table is written)
    // halo tile: NPIX pixels x 4 channel quads
    for (int i = gtid; i < NPIX * (CK / 4); i += GT) {
      const int pix = i / (CK / 4), q = i % (CK / 4);
      const int hh = h0 - 1 + pix / WP, ww = w0 - 1 + pix % WP;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (hh >= 0 && hh < H && ww >= 0 && ww < W) {
        const int c = c0 + q * 4;
        v = __ldcs(reinterpret_cast<const float4*>(x + ((size_t)n * HW + (size_t)hh * W + ww) * C + c));
        v.x = silu_f(fmaf(v.x, s_scale[c], s_shift[c])), v.y = silu_f(fmaf(v.y, s_scale[c + 1], s_shift[c + 1]));
        v.z = silu_f(fmaf(v.z, s_scale[c + 2], s_shift[c + 2])), v.w = silu_f(fmaf(v.w, s_scale[c + 3], s_shift[c + 3]));
      }
      s_act[q * NPIX + pix] = v;  // zero outside the image == the conv's zero padding of the NORMALISED tensor
    }
    for (int i = gtid; i < 9 * COUT * (CK / 4); i += GT) {
      const int q = i % (CK / 4), o = (i / (CK / 4)) % COUT, tap = i / ((CK / 4) * COUT);
      s_w[i] = *reinterpret_cast<const float4*>(wp + ((size_t)o * 9 + tap) * C + c0 + q * 4);
    }
    __syncthreads();
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int pix = (ty + tap / 3) * WP + tx + tap % 3;
#pragma unroll
      for (int q = 0; q < CK / 4; ++q) {
        const float4 a = s_act[q * NPIX + pix];
#pragma unroll
        for (int o = 0; o < COUT; ++o) {
          const float4 wv = s_w[(tap * COUT + o) * (CK / 4) + q];
          acc[o] = fmaf(a.x, wv.x, fmaf(a.y, wv.y, fmaf(a.z, wv.z, fmaf(a.w, wv.w, acc[o]))));
        }
      }
    }
  }
  if (KS > 1) {
    // partial sums of the groups -> shared memory (over the tiles, which are dead now), added in group order by group 0
    __syncthreads();
    float* s_red = sm + 2 * C;  // [KS][COUT][GT]
#pragma unroll
    for (int o = 0; o < COUT; ++o) s_red[(ks * COUT + o) * GT + gtid] = acc[o];
    __syncthreads();
    if (ks == 0) {
#pragma unroll
      for (int o = 0; o < COUT; ++o) {
        float a = s_red[o * GT + gtid];
        for (int k = 1; k < KS; ++k) a += s_red[(k * COUT + o) * GT + gtid];
        acc[o] = a;
      }
    }
  }
  const int h = h0 + ty, w = w0 + tx;
  if (ks == 0 && h < H && w < W) {
#pragma unroll
    for (int o = 0; o < COUT; ++o) y[((size_t)n * COUT + o) * HW + (size_t)h * W + w] = acc[o] + b[o];
  }
}
void conv3x3_small_cout_launch(const float* x, int n, int H, int W, int C, const double* sums, const float* gamma,
                               const float* beta, float eps, const float* w_packed, const float* b, int Cout,
                               float* y_nchw, cudaStream_t st) {
  SDB_CHECK(C % 16 == 0, "conv3x3_small_cout: channels must be a multiple of 16");
  // too few 8-row tiles to fill the machine -> 2-row tiles, 32 channels per round and group, the channel chunks split over
  // KS = 5 or 4 groups of two warps (10 / 8 warps per CTA; 320 = 10 x 32 and 512 = 16 x 32 channels)
  const bool small = (long long)ceil_div(W, 32) * ceil_div(H, 8) * n < 2 * 148 && C % 32 == 0;
  const int ksplit = !small ? 1 : ((C / 32) % 5 == 0 ? 5 : ((C / 32) % 4 == 0 ? 4 : 1));
  const int th = small ? 2 : 8, ck = small ? 32 : 16;
  dim3 grid(ceil_div(W, 32), ceil_div(H, th), n), block(32 * th * ksplit);
  auto smem = [&](int cout) {
    return (size_t)(2 * C + std::max(ksplit * (ck * (th + 2) * 34 + 9 * cout * ck), ksplit * cout * 32 * th)) * sizeof(float);
  };
#define SDB_SMALL_KS(CO, KSV)                                                                                                       \
  {                                                                                                                                 \
    static DeviceOnce once;                                                                                                         \
    if (once.first())                                                                                                               \
      SDB_CUDA(cudaFuncSetAttribute(conv3x3_small_cout_kernel<CO, 2, 32, KSV>, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                    160 * 1024));                                                                                   \
    SDB_CHECK(smem(CO) <= 160 * 1024, "conv3x3_small_cout: shared memory");                                                         \
    launch_k(conv3x3_small_cout_kernel<CO, 2, 32, KSV>, grid, block, smem(CO), st, x, H, W, C, sums, gamma, beta, eps, w_packed, b, \
             y_nchw);                                                                                                               \
  }
#define SDB_SMALL_CONV(CO)                                                                                                          \
  if (small) {                                                                                                                      \
    if (ksplit == 5) SDB_SMALL_KS(CO, 5) else if (ksplit == 4) SDB_SMALL_KS(CO, 4) else SDB_SMALL_KS(CO, 1)                          \
  } else                                                                                                                            \
    launch_k(conv3x3_small_cout_kernel<CO, 8, 16>, grid, block, smem(CO), st, x, H, W, C, sums, gamma, beta, eps, w_packed, b, y_nchw)
  if (Cout == 4) {
    SDB_SMALL_CONV(4);
  } else if (Cout == 3) {
    SDB_SMALL_CONV(3);
  } else if (Cout == 8) {
    SDB_SMALL_CONV(8);
  } else {
    throw Error("conv3x3_small_cout: Cout must be 3, 4 or 8");
  }
#undef SDB_SMALL_CONV
#undef SDB_SMALL_KS
  SDB_CUDA(cudaGetLastError());
}

// quant_conv (1x1, 8 -> 8) followed by the slice [0..4) of Autoencoder::encode_image (autoencoder/mod.rs:60-66): NCHW in/out
__global__ void quant_conv_slice_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                                        int HW, float* __restrict__ y) {
  const int n = blockIdx.y;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += gridDim.x * blockDim.x) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = x[((size_t)n * 8 + j) * HW + p];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float acc = b[c];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc += w[c * 8 + j] * v[j];
      y[((size_t)n * 4 + c) * HW + p] = acc;
    }
  }
}
void quant_conv_slice_launch(const float* x, const float* w, const float* b, int n, int HW, float* y, cudaStream_t st) {
  dim3 grid(std::min(ceil_div(HW, 256), 1024), n);
  quant_conv_slice_kernel<<<grid, 256, 0, st>>>(x, w, b, HW, y);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ time embedding + GEMV
// y[N] = act(x[K] W[K][N] + b); a block owns 32 outputs, 8 k-slices reduced through smem.
// t_dev != null: x is the sinusoidal timestep embedding (reference unet/mod.rs:24-29), K must be 320.
__global__ void __launch_bounds__(256)
gemv_kernel(const float* __restrict__ x, const int* __restrict__ t_dev, const float* __restrict__ W,
            const float* __restrict__ b, int K, int N, int silu, float* __restrict__ y) {
  pdl_enter();
  __shared__ float s_part[8][32];
  __shared__ float s_x[1280];
  if (t_dev) {
    const int t = *t_dev;
    for (int i = threadIdx.x; i < 160; i += blockDim.x) {
      // freqs = exp(arange(half) * (-ln(10000)/half)); args = t*freqs; [cos | sin]
      const float f = expf((float)i * (float)(-9.210340371976184 / 160.0));
      const float a = (float)t * f;
      s_x[i] = cosf(a);
      s_x[160 + i] = sinf(a);
    }
  } else {
    for (int i = threadIdx.x; i < K; i += blockDim.x) s_x[i] = x[i];
  }
  __syncthreads();
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ks = threadIdx.x >> 5;  // 0..7
  float acc = 0.f;
  if (col < N)
    for (int k = ks; k < K; k += 8) acc += s_x[k] * W[(size_t)k * N + col];
  s_part[ks][threadIdx.x & 31] = acc;
  __syncthreads();
  if (ks == 0 && col < N) {
    float s = b ? b[col] : 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += s_part[j][threadIdx.x & 31];
    y[col] = silu ? silu_f(s) : s;
  }
}
void gemv_launch(const float* x, const float* W, const float* b, int K, int N, float* y, cudaStream_t st) {
  SDB_CHECK(K <= 1280, "gemv K");
  launch_k(gemv_kernel, dim3(ceil_div(N, 32)), dim3(256), 0, st, x, (const int*)nullptr, W, b, K, N, 0, y);
  SDB_CUDA(cudaGetLastError());
}
// emb_silu = silu(lin2(silu(lin1(timestep_embedding(t)))))  — two multi-CTA GEMVs (was one CTA: 140 us)
void time_embed_launch(const int* t, const float* w1, const float* b1, const float* w2, const float* b2, float* hidden,
                       float* emb_silu, cudaStream_t st) {
  launch_k(gemv_kernel, dim3(40), dim3(256), 0, st, (const float*)nullptr, t, w1, b1, 320, 1280, 1, hidden);
  launch_k(gemv_kernel, dim3(40), dim3(256), 0, st, (const float*)hidden, (const int*)nullptr, w2, b2, 1280, 1280, 1, emb_silu);
  SDB_CUDA(cudaGetLastError());
}

// Time embedding for ALL timesteps of a sampling schedule in one pass (the rows depend on t alone: sample_latent computes them once
// per call instead of once per step; the weights of the 22 lin_embed layers, 103 MB of fp32, stream once per R rows instead of
// once per step). Same arithmetic, in the same order, as gemv_kernel: the rows are bit-identical to the per-step path.
//   y[row][N] = act(x[row][K] W[K][N] + b),  row = blockIdx.y * R + r
// t_embed != null: x is the sinusoidal embedding of t_embed[row] (K = 320). t_rowmap != null: output row index = t_rowmap[row].
template <int R>
__global__ void __launch_bounds__(256)
gemv_rows_kernel(const float* __restrict__ x, const int* __restrict__ t_embed, const int* __restrict__ t_rowmap, int rows,
                 const float* __restrict__ W, const float* __restrict__ b, int K, int N, int silu, float* __restrict__ y,
                 long long y_stride) {
  pdl_enter();
  __shared__ float s_part[R][8][32];
  __shared__ float s_x[R][1280];
  const int r0 = blockIdx.y * R, nr = min(R, rows - r0);
  for (int r = 0; r < nr; ++r) {
    if (t_embed) {
      const int t = t_embed[r0 + r];
      for (int i = threadIdx.x; i < 160; i += blockDim.x) {
        const float f = expf((float)i * (float)(-9.210340371976184 / 160.0));
        const float a = (float)t * f;
        s_x[r][i] = cosf(a);
        s_x[r][160 + i] = sinf(a);
      }
    } else {
      for (int i = threadIdx.x; i < K; i += blockDim.x) s_x[r][i] = x[(size_t)(r0 + r) * K + i];
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int col = blockIdx.x * 32 + lane;
  const int ks = threadIdx.x >> 5;  // 0..7
  float acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = 0.f;
  if (col < N)
    for (int k = ks; k < K; k += 8) {
      const float w = W[(size_t)k * N + col];
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] += s_x[r][k] * w;  // rows >= nr read stale shared memory and are never stored
    }
#pragma unroll
  for (int r = 0; r < R; ++r) s_part[r][ks][lane] = acc[r];
  __syncthreads();
  if (ks == 0 && col < N) {
    for (int r = 0; r < nr; ++r) {
      float s = b ? b[col] : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) s += s_part[r][j][lane];
      const long long orow = t_rowmap ? t_rowmap[r0 + r] : (r0 + r);
      y[orow * y_stride + col] = silu ? silu_f(s) : s;
    }
  }
}
// rows of emb_all are indexed by the TIMESTEP VALUE (emb_all[t][N]): the in-graph selection needs no step counter
void time_embed_rows_launch(const int* t_dev, int rows, const float* w1, const float* b1, const float* w2, const float* b2,
                            const float* w_all, const float* b_all, int n_all, float* hidden, float* emb_silu, float* emb_all,
                            cudaStream_t st) {
  constexpr int R = 5;
  const dim3 gy(40, ceil_div(rows, R));
  launch_k(gemv_rows_kernel<R>, gy, dim3(256), 0, st, (const float*)nullptr, t_dev, (const int*)nullptr, rows, w1, b1, 320, 1280, 1,
           hidden, (long long)1280);
  launch_k(gemv_rows_kernel<R>, gy, dim3(256), 0, st, (const float*)hidden, (const int*)nullptr, (const int*)nullptr, rows, w2, b2,
           1280, 1280, 1, emb_silu, (long long)1280);
  launch_k(gemv_rows_kernel<R>, dim3(ceil_div(n_all, 32), ceil_div(rows, R)), dim3(256), 0, st, (const float*)emb_silu,
           (const int*)nullptr, t_dev, rows, w_all, b_all, 1280, n_all, 0, emb_all, (long long)n_all);
  SDB_CUDA(cudaGetLastError());
}
// out[N] = emb_all[*t_dev][N]: the one launch of the UNet step graph that replaces the three GEMVs
__global__ void __launch_bounds__(256)
emb_select_kernel(const float* __restrict__ emb_all, const int* __restrict__ t_dev, int N, float* __restrict__ out) {
  pdl_enter();
  const float4* src = reinterpret_cast<const float4*>(emb_all + (size_t)(*t_dev) * N);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N / 4; i += gridDim.x * blockDim.x)
    reinterpret_cast<float4*>(out)[i] = src[i];
}
void emb_select_launch(const float* emb_all, const int* t_dev, int N, float* out, cudaStream_t st) {
  SDB_CHECK(N % 4 == 0, "emb_select: N must be a multiple of 4");
  launch_k(emb_select_kernel, dim3(ceil_div(N / 4, 256)), dim3(256), 0, st, emb_all, t_dev, N, out);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ CLIP token + position embedding
// x[s][l][:] = E[tok[s][l]] + Pos[l] for l < L, zero rows up to Lp (reference clip/mod.rs:62-68)
__global__ void embed_tokens_kernel(const int* __restrict__ tok, const float* __restrict__ E, const float* __restrict__ Pos,
                                    int L, int Lp, int D, int vocab, float* __restrict__ x) {
  pdl_enter();
  const int row = blockIdx.x;  // s*Lp + l
  const int s = row / Lp, l = row % Lp;
  float4* dst = reinterpret_cast<float4*>(x + (size_t)row * D);
  if (l >= L) {
    for (int i = threadIdx.x; i < D / 4; i += blockDim.x) dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  int id = tok[s * L + l];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  const float4* e = reinterpret_cast<const float4*>(E + (size_t)id * D);
  const float4* pp = reinterpret_cast<const float4*>(Pos + (size_t)l * D);
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) {
    const float4 a = e[i], b = pp[i];
    dst[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}
void embed_tokens_launch(const int* tok, const float* E, const float* Pos, int n, int L, int Lp, int D, int vocab, float* x,
                         cudaStream_t st) {
  launch_k(embed_tokens_kernel, dim3(n * Lp), dim3(192), 0, st, tok, E, Pos, L, Lp, D, vocab, x);
}

// y = a + b (merged conv biases at finalize)
__global__ void add_vec_kernel(const float* __restrict__ a, const float* __restrict__ b, int n, float* __restrict__ y) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = a[i] + b[i];
}
void add_vec_launch(const float* a, const float* b, int n, float* y, cudaStream_t st) {
  add_vec_kernel<<<ceil_div(n, 256), 256, 0, st>>>(a, b, n, y);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ sampler elementwise
__global__ void cfg_ddim_kernel(const float* __restrict__ eu, const float* __restrict__ ec, float* __restrict__ lat,
                                long long count, float scale, float sqrt_1m_at, float sqrt_at, float sqrt_aprev,
                                float dir_coef) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    const float u = eu[i], c = ec[i];
    const float pred = u + (c - u) * scale;               // stablediffusion/mod.rs:190-191
    const float x0 = (lat[i] - pred * sqrt_1m_at) / sqrt_at;  // :152
    const float nl = x0 * sqrt_aprev + pred * dir_coef;   // :153-155 (sigma = 0)
    lat[i] = nl;
    lat[i + count] = nl;  // the UNet input batch holds the latent twice (uncond half | cond half)
  }
}
void cfg_ddim_launch(const float* eps_u, const float* eps_c, float* latent, long long count, float scale,
                     float sqrt_one_minus_at, float sqrt_at, float sqrt_aprev, float dir_coef, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  launch_k(cfg_ddim_kernel, dim3(grid), dim3(256), 0, st, eps_u, eps_c, latent, count, scale, sqrt_one_minus_at, sqrt_at, sqrt_aprev, dir_coef);
  SDB_CUDA(cudaGetLastError());
}

__global__ void cfg_combine_kernel(const float* __restrict__ eu, const float* __restrict__ ec, long long count, float scale,
                                   float* __restrict__ pred) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
    pred[i] = eu[i] + (ec[i] - eu[i]) * scale;  // stablediffusion/mod.rs:190-191
}
void cfg_combine_launch(const float* eps_u, const float* eps_c, long long count, float scale, float* pred, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  cfg_combine_kernel<<<grid, 256, 0, st>>>(eps_u, eps_c, count, scale, pred);
  SDB_CUDA(cudaGetLastError());
}

__global__ void to_rgb8_kernel(const float* __restrict__ img, int HW, long long total, uint8_t* __restrict__ rgb) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % 3);
    const long long r = i / 3;
    const int p = int(r % HW);
    const long long n = r / HW;
    float v = img[(n * 3 + c) * HW + p];
    v = (v + 1.0f) / 2.0f * 255.0f;             // stablediffusion/mod.rs:79-84
    // :96  v.to_f64().min(255.0).max(0.0) as u8  (NaN -> min gives 255)
    float m = (v != v) ? 255.0f : fminf(v, 255.0f);
    m = fmaxf(m, 0.0f);
    rgb[i] = (uint8_t)m;                        // truncation toward zero
  }
}
void to_rgb8_launch(const float* img_nchw, int n, int H, int W, uint8_t* rgb, cudaStream_t st) {
  const long long total = (long long)n * 3 * H * W;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  to_rgb8_kernel<<<grid, 256, 0, st>>>(img_nchw, H * W, total, rgb);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ img2img / inpainting (DESIGN.md §7 row f5)
// u8 HWC [n][H][W][3] -> fp32 planes [n][4][H][W] (fourth plane zero, the layout of the encoder's Cin = 4 conv_in):
// x = fl(fl(v * fl32(2/255)) - 1), no FMA, so numpy fp32 reproduces it bit for bit
__global__ void rgb8_to_planes4_kernel(const uint8_t* __restrict__ rgb, int HW, long long total, float* __restrict__ img4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = int(i % HW);
    const long long r = i / HW;
    const int c = int(r % 4);
    const long long n = r / 4;
    img4[i] = c < 3 ? __fsub_rn(__fmul_rn((float)rgb[(n * HW + p) * 3 + c], (float)(2.0 / 255.0)), 1.0f) : 0.0f;
  }
}
void rgb8_to_planes4_launch(const uint8_t* rgb, int n, int H, int W, float* img4, cudaStream_t st) {
  const long long total = (long long)n * 4 * H * W;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  rgb8_to_planes4_kernel<<<grid, 256, 0, st>>>(rgb, H * W, total, img4);
  SDB_CUDA(cudaGetLastError());
}

// latent cell (y, x) is repainted when any pixel of its 8x8 block is: m[n][H][W] = max over the block of (mask != 0)
__global__ void latent_mask_kernel(const uint8_t* __restrict__ mask, int H, int W, long long total, uint8_t* __restrict__ m) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = int(i % W);
    const long long r = i / W;
    const int y = int(r % H);
    const long long n = r / H;
    const uint8_t* blk = mask + ((n * 8 * H + 8 * y) * 8 * W + 8 * x);
    uint32_t any = 0;
#pragma unroll
    for (int dy = 0; dy < 8; ++dy)
#pragma unroll
      for (int dx = 0; dx < 8; ++dx) any |= blk[(size_t)dy * 8 * W + dx];
    m[i] = any ? 1 : 0;
  }
}
void latent_mask_launch(const uint8_t* mask, int n, int H, int W, uint8_t* m, cudaStream_t st) {
  const long long total = (long long)n * H * W;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  latent_mask_kernel<<<grid, 256, 0, st>>>(mask, H, W, total, m);
  SDB_CUDA(cudaGetLastError());
}

__global__ void scale_kernel(float* __restrict__ x, long long count, float s) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
    x[i] = __fmul_rn(x[i], s);
}
void scale_launch(float* x, long long count, float s, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  scale_kernel<<<grid, 256, 0, st>>>(x, count, s);
  SDB_CUDA(cudaGetLastError());
}

// x_t0 = fl(fl(a * x0) + fl(b * eps)) into both halves of the batch-2n UNet input (as cfg_ddim_kernel writes them)
__global__ void noise_latent_kernel(const float* __restrict__ x0, const float* __restrict__ eps, long long count, float a, float b,
                                    float* __restrict__ lat) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    const float v = __fadd_rn(__fmul_rn(a, x0[i]), __fmul_rn(b, eps[i]));
    lat[i] = v;
    lat[i + count] = v;
  }
}
void noise_latent_launch(const float* x0, const float* eps, long long count, float a, float b, float* latent, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  noise_latent_kernel<<<grid, 256, 0, st>>>(x0, eps, count, a, b, latent);
  SDB_CUDA(cudaGetLastError());
}

// cfg_ddim_kernel's update, then the kept cells (m == 0) are selected from the known image noised to a_prev:
// known = fl(fl(sqrt(a_prev) * x0) + fl(sqrt(1 - a_prev) * eps)) — the same two coefficients as the update's
__global__ void cfg_ddim_blend_kernel(const float* __restrict__ eu, const float* __restrict__ ec, float* __restrict__ lat,
                                      long long count, float scale, float sqrt_1m_at, float sqrt_at, float sqrt_aprev,
                                      float dir_coef, const float* __restrict__ x0, const float* __restrict__ eps,
                                      const uint8_t* __restrict__ m, int HW) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    const float u = eu[i], c = ec[i];
    const float pred = u + (c - u) * scale;               // stablediffusion/mod.rs:190-191
    const float px0 = (lat[i] - pred * sqrt_1m_at) / sqrt_at;  // :152
    float nl = px0 * sqrt_aprev + pred * dir_coef;        // :153-155 (sigma = 0)
    const long long cell = (i / (4LL * HW)) * HW + i % HW;
    if (!m[cell]) nl = __fadd_rn(__fmul_rn(sqrt_aprev, x0[i]), __fmul_rn(dir_coef, eps[i]));
    lat[i] = nl;
    lat[i + count] = nl;
  }
}
void cfg_ddim_blend_launch(const float* eps_u, const float* eps_c, float* latent, long long count, float scale,
                           float sqrt_one_minus_at, float sqrt_at, float sqrt_aprev, float dir_coef, const float* x0,
                           const float* eps, const uint8_t* m, int HW, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  launch_k(cfg_ddim_blend_kernel, dim3(grid), dim3(256), 0, st, eps_u, eps_c, latent, count, scale, sqrt_one_minus_at, sqrt_at,
           sqrt_aprev, dir_coef, x0, eps, m, HW);
  SDB_CUDA(cudaGetLastError());
}

// to_rgb8_kernel's conversion, except that pixels with mask == 0 are copied from the source image unchanged
__global__ void to_rgb8_paste_kernel(const float* __restrict__ img, int HW, long long total, const uint8_t* __restrict__ src,
                                     const uint8_t* __restrict__ mask, uint8_t* __restrict__ rgb) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / 3;
    if (!mask[r]) {
      rgb[i] = src[i];
      continue;
    }
    const int c = int(i % 3);
    const int p = int(r % HW);
    const long long n = r / HW;
    float v = img[(n * 3 + c) * HW + p];
    v = (v + 1.0f) / 2.0f * 255.0f;             // stablediffusion/mod.rs:79-84
    float mm = (v != v) ? 255.0f : fminf(v, 255.0f);
    mm = fmaxf(mm, 0.0f);
    rgb[i] = (uint8_t)mm;
  }
}
void to_rgb8_paste_launch(const float* img_nchw, int n, int H, int W, const uint8_t* src_rgb, const uint8_t* mask, uint8_t* rgb,
                          cudaStream_t st) {
  const long long total = (long long)n * 3 * H * W;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  to_rgb8_paste_kernel<<<grid, 256, 0, st>>>(img_nchw, H * W, total, src_rgb, mask, rgb);
  SDB_CUDA(cudaGetLastError());
}


__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x85EBCA6Bu;
  x ^= x >> 13;
  x *= 0xC2B2AE35u;
  x ^= x >> 16;
  return x;
}
// element i of the seeded N(0,1) stream keyed by (k0, k1): Box-Muller on two hashed uniforms. randn_kernel and
// cfg_ddim_eta_kernel both draw through this one function, so an in-kernel draw equals randn_launch's output bit for bit.
__device__ __forceinline__ float randn_at(long long i, uint32_t k0, uint32_t k1) {
  const uint32_t a = mix32((uint32_t)i ^ k0), b = mix32(((uint32_t)i * 0x9E3779B9u) ^ k1);
  const float u1 = ((a >> 8) + 1) * (1.0f / 16777216.0f);  // (0,1]
  const float u2 = (b >> 8) * (1.0f / 16777216.0f);
  return sqrtf(-2.0f * logf(u1)) * cosf(6.283185307179586f * u2);
}
static inline uint32_t randn_key0(uint64_t seed) { return (uint32_t)seed * 2654435761u + 1u; }
static inline uint32_t randn_key1(uint64_t seed) { return (uint32_t)(seed >> 32) ^ 0x5bd1e995u; }

__global__ void randn_kernel(float* __restrict__ x, long long count, uint32_t k0, uint32_t k1) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
    x[i] = randn_at(i, k0, k1);
}
void randn_launch(float* x, long long count, uint64_t seed, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  randn_kernel<<<grid, 256, 0, st>>>(x, count, randn_key0(seed), randn_key1(seed));
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ selectable samplers (DESIGN.md §7 row f6)
// Both kernels round once per operation (__f*_rn: no contraction), in the order of oracle/sampler_oracle.py's
// ddim_update_f32 / dpmpp_2m_update_f32, so a numpy f32 replay of a step matches the device bit for bit.
__device__ __forceinline__ void cfg_x0_rn(float u, float c, float x, float scale, float sqrt_1m_at, float sqrt_at, float& pred,
                                          float& x0) {
  pred = __fadd_rn(u, __fmul_rn(__fsub_rn(c, u), scale));            // stablediffusion/mod.rs:190-191
  x0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(pred, sqrt_1m_at)), sqrt_at);  // :152
}

// DDIM with eta > 0: x' = x0*sqrt_anext + pred*dir + sigma*z (mod.rs:153-155 with sigma != 0). z is z_explicit[i], or element i
// of the seeded stream (k0, k1) when z_explicit is null. sigma == 0 (the last step) reads no noise at all.
__global__ void cfg_ddim_eta_kernel(const float* __restrict__ eu, const float* __restrict__ ec, float* __restrict__ lat,
                                    long long count, float scale, float sqrt_1m_at, float sqrt_at, float sqrt_anext, float dir,
                                    float sigma, const float* __restrict__ z_explicit, uint32_t k0, uint32_t k1) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    float pred, x0;
    cfg_x0_rn(eu[i], ec[i], lat[i], scale, sqrt_1m_at, sqrt_at, pred, x0);
    float nl = __fadd_rn(__fmul_rn(x0, sqrt_anext), __fmul_rn(pred, dir));
    if (sigma != 0.0f) nl = __fadd_rn(nl, __fmul_rn(sigma, z_explicit ? z_explicit[i] : randn_at(i, k0, k1)));
    lat[i] = nl;
    lat[i + count] = nl;
  }
}
void cfg_ddim_eta_launch(const float* eps_u, const float* eps_c, float* latent, long long count, float scale,
                         float sqrt_one_minus_at, float sqrt_at, float sqrt_anext, float dir, float sigma, const float* z,
                         uint64_t z_seed, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  launch_k(cfg_ddim_eta_kernel, dim3(grid), dim3(256), 0, st, eps_u, eps_c, latent, count, scale, sqrt_one_minus_at, sqrt_at,
           sqrt_anext, dir, sigma, z, randn_key0(z_seed), randn_key1(z_seed));
  SDB_CUDA(cudaGetLastError());
}

// DPM-Solver++(2M): KIND 0 = first order (D = x0), 1 = second order (D = x0*w0 - hist*w1), 2 = final (x' = x0).
// x' = x*ratio - D*coef; hist [count] holds x0 of the previous step and receives this step's. The first-order and final
// variants never read hist (before step 0 it is uninitialised, and 0*NaN is NaN); the final one does not write it either.
template <int KIND>
__global__ void cfg_dpmpp2m_kernel(const float* __restrict__ eu, const float* __restrict__ ec, float* __restrict__ lat,
                                   float* __restrict__ hist, long long count, float scale, float sqrt_1m_at, float sqrt_at,
                                   float ratio, float coef, float w0, float w1) {
  pdl_enter();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    const float x = lat[i];
    float pred, x0;
    cfg_x0_rn(eu[i], ec[i], x, scale, sqrt_1m_at, sqrt_at, pred, x0);
    float nl = x0;
    if (KIND != 2) {
      const float D = KIND == 0 ? x0 : __fsub_rn(__fmul_rn(x0, w0), __fmul_rn(hist[i], w1));
      nl = __fsub_rn(__fmul_rn(x, ratio), __fmul_rn(D, coef));
      hist[i] = x0;
    }
    lat[i] = nl;
    lat[i + count] = nl;
  }
}
void cfg_dpmpp2m_launch(int kind, const float* eps_u, const float* eps_c, float* latent, float* hist, long long count, float scale,
                        float sqrt_one_minus_at, float sqrt_at, float ratio, float coef, float w0, float w1, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  auto k = kind == 0 ? cfg_dpmpp2m_kernel<0> : kind == 1 ? cfg_dpmpp2m_kernel<1> : cfg_dpmpp2m_kernel<2>;
  launch_k(k, dim3(grid), dim3(256), 0, st, eps_u, eps_c, latent, hist, count, scale, sqrt_one_minus_at, sqrt_at, ratio, coef,
           w0, w1);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ weight packing
__device__ __forceinline__ void split_store1(float f, __half* hi, __half* lo, size_t o) {
  const __half h = __float2half_rn(f);
  hi[o] = h;
  if (lo) lo[o] = __float2half_rn(f - __half2float(h));
}
__global__ void pack_conv_kernel(const float* __restrict__ w, int Cout, int Cin, int kk, __half* hi, __half* lo) {
  const long long total = (long long)Cout * kk * Cin;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % Cin);
    const long long r = i / Cin;
    const int tap = int(r % kk);
    const long long co = r / kk;
    split_store1(w[(co * Cin + c) * kk + tap], hi, lo, (size_t)i);
  }
}
void pack_conv_launch(const float* w, int Cout, int Cin, int ksize, Half2Ptr out, cudaStream_t st) {
  const long long total = (long long)Cout * ksize * ksize * Cin;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  pack_conv_kernel<<<grid, 256, 0, st>>>(w, Cout, Cin, ksize * ksize, out.hi, out.lo);
  SDB_CUDA(cudaGetLastError());
}

// nearest-2x upsample folded into the following 3x3 conv: output phase (a,b) in {0,1}^2 sees a 2x2 window of
// the low-res source; window tap (i,j) accumulates the 3x3 taps that land on the same source pixel:
//   a=0: rows {0} -> i=0, {1,2} -> i=1 ;  a=1: rows {0,1} -> i=0, {2} -> i=1   (same for columns)
__global__ void pack_conv_up2_kernel(const float* __restrict__ w, int Cout, int Cin, __half* hi, __half* lo) {
  const long long total = (long long)4 * Cout * 4 * Cin;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % Cin);
    long long r = i / Cin;
    const int wt = int(r % 4);
    r /= 4;
    const int co = int(r % Cout);
    const int phase = int(r / Cout);
    const int a = phase >> 1, b = phase & 1, ti = wt >> 1, tj = wt & 1;
    float acc = 0.f;
    for (int kh = 0; kh < 3; ++kh) {
      const int ii = (a == 0) ? (kh == 0 ? 0 : 1) : (kh == 2 ? 1 : 0);
      if (ii != ti) continue;
      for (int kw = 0; kw < 3; ++kw) {
        const int jj = (b == 0) ? (kw == 0 ? 0 : 1) : (kw == 2 ? 1 : 0);
        if (jj != tj) continue;
        acc += w[(((size_t)co * Cin + c) * 3 + kh) * 3 + kw];
      }
    }
    split_store1(acc, hi, lo, (size_t)i);
  }
}
void pack_conv_up2_launch(const float* w, int Cout, int Cin, Half2Ptr out, cudaStream_t st) {
  const long long total = (long long)16 * Cout * Cin;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  pack_conv_up2_kernel<<<grid, 256, 0, st>>>(w, Cout, Cin, out.hi, out.lo);
  SDB_CUDA(cudaGetLastError());
}

__global__ void pack_linear_kernel(const float* __restrict__ w, int in, int out, int ldw, int col0, __half* hi, __half* lo,
                                   int row_offset, const float* __restrict__ in_scale) {
  // tiled transpose [in][out] -> [out][in]; in_scale (optional) multiplies input feature i: a LayerNorm's gamma folded into
  // the weights of the GEMM that consumes the normalised tensor
  __shared__ float tile[32][33];
  const int o0 = blockIdx.x * 32, i0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int i = i0 + r, o = o0 + threadIdx.x;
    tile[r][threadIdx.x] = (i < in && o < out) ? w[(size_t)i * ldw + col0 + o] * (in_scale ? in_scale[i] : 1.0f) : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int o = o0 + r, i = i0 + threadIdx.x;
    if (o < out && i < in) split_store1(tile[threadIdx.x][r], hi, lo, (size_t)(row_offset + o) * in + i);
  }
}
void pack_linear_launch(const float* w, int in, int out, Half2Ptr dst, int row_offset, cudaStream_t st, int ldw,
                        int col0, const float* in_scale) {
  dim3 grid(ceil_div(out, 32), ceil_div(in, 32)), block(32, 8);
  pack_linear_kernel<<<grid, block, 0, st>>>(w, in, out, ldw ? ldw : out, col0, dst.hi, dst.lo, row_offset, in_scale);
  SDB_CUDA(cudaGetLastError());
}

// row sums of a packed fp16 matrix [rows][K]: s_hi[r] = sum_k hi[r][k], s_full[r] = sum_k (hi + lo)[r][k] (fp32 accumulation
// in a fixed order: one warp per row, lanes stride K, xor-tree) — the "u" vector of a LayerNorm folded into a GEMM: it must be
// the sum of exactly the values the tensor cores multiply, or the mean would not cancel
__global__ void __launch_bounds__(256) rowsum_f16_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, int rows,
                                                         int K, float* __restrict__ s_hi, float* __restrict__ s_full) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  float a = 0.f, b = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float h = __half2float(hi[(size_t)row * K + k]);
    a += h;
    b += h + (lo ? __half2float(lo[(size_t)row * K + k]) : 0.f);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o), b += __shfl_xor_sync(0xffffffffu, b, o);
  if (lane == 0) {
    if (s_hi) s_hi[row] = a;
    if (s_full) s_full[row] = b;
  }
}
void rowsum_f16_launch(Half2Ptr m, int rows, int K, float* s_hi, float* s_full, cudaStream_t st) {
  rowsum_f16_kernel<<<ceil_div(rows, 8), 256, 0, st>>>(m.hi, m.lo, rows, K, s_hi, s_full);
  SDB_CUDA(cudaGetLastError());
}

__global__ void pack_geglu_kernel(const float* __restrict__ w, const float* __restrict__ b, int in, int h4, int half_tile,
                                  __half* hi, __half* lo, float* bias_packed, const float* __restrict__ in_scale) {
  // packed row pr in [0, 2*h4): tile j = pr / (2*half_tile); within tile q = pr % (2*half_tile);
  // q < half_tile -> x column j*half_tile + q ; else gate column h4 + j*half_tile + (q - half_tile)
  const long long total = (long long)2 * h4 * in;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int i = int(idx % in);
    const int pr = int(idx / in);
    const int j = pr / (2 * half_tile), q = pr % (2 * half_tile);
    const int col = (q < half_tile) ? j * half_tile + q : h4 + j * half_tile + (q - half_tile);
    split_store1(w[(size_t)i * (2 * h4) + col] * (in_scale ? in_scale[i] : 1.0f), hi, lo, (size_t)idx);
    if (i == 0 && bias_packed) bias_packed[pr] = b[col];
  }
}
void pack_geglu_launch(const float* w, const float* b, int in, int h4, int half_tile, Half2Ptr dst, float* bias_packed,
                       cudaStream_t st, const float* in_scale) {
  const long long total = (long long)2 * h4 * in;
  int grid = (int)((total + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  pack_geglu_kernel<<<grid, 256, 0, st>>>(w, b, in, h4, half_tile, dst.hi, dst.lo, bias_packed, in_scale);
  SDB_CUDA(cudaGetLastError());
}

__global__ void pack_small_cout_kernel(const float* __restrict__ w, int Cout, int Cin, float* __restrict__ out) {
  const int total = Cout * 9 * Cin;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c = i % Cin, tap = (i / Cin) % 9, co = i / (9 * Cin);
    out[i] = w[((size_t)co * Cin + c) * 9 + tap];
  }
}
void pack_small_cout_launch(const float* w, int Cout, int Cin, float* out, cudaStream_t st) {
  pack_small_cout_kernel<<<ceil_div(Cout * 9 * Cin, 256), 256, 0, st>>>(w, Cout, Cin, out);
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ row softmax (VAE attention, 1 head, d = 512)
// P[r][:] = softmax(S[r][:] * scale) -> fp16 hi(/lo); one CTA per row, row kept in registers
template <int PER>
__global__ void __launch_bounds__(256)
softmax_rows_kernel(const float* __restrict__ S, int cols, float scale_log2, __half* __restrict__ hi,
                    __half* __restrict__ lo) {
  __shared__ float red[8];
  const size_t row = blockIdx.x;
  const float* sr = S + row * cols;
  float v[PER];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int i = threadIdx.x + k * 256;
    v[k] = i < cols ? sr[i] * scale_log2 : -INFINITY;
    mx = fmaxf(mx, v[k]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) mx = fmaxf(mx, red[k]);
  __syncthreads();
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    v[k] = exp2f(v[k] - mx);
    sum += v[k];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  sum = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) sum += red[k];
  const float inv = 1.0f / sum;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int i = threadIdx.x + k * 256;
    if (i < cols) split_store1(v[k] * inv, hi, lo, row * cols + i);
  }
}
void softmax_rows_launch(const float* S, long long rows, int cols, float scale, Half2Ptr out, cudaStream_t st) {
  const float sl2 = scale * 1.4426950408889634f;
  if (cols <= 4096)
    softmax_rows_kernel<16><<<(unsigned)rows, 256, 0, st>>>(S, cols, sl2, out.hi, out.lo);
  else if (cols <= 9216)
    softmax_rows_kernel<36><<<(unsigned)rows, 256, 0, st>>>(S, cols, sl2, out.hi, out.lo);
  else
    throw Error("softmax_rows: row too long");
  SDB_CUDA(cudaGetLastError());
}

// ============================================================ synthetic weights
__global__ void synth_fill_kernel(float* __restrict__ dst, long long count, uint32_t key, float bound, float offset) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t h = mix32((uint32_t)i ^ key);
    const float u = (float)(h >> 8) * (1.0f / 16777216.0f);
    // (u*2 - 1) is exact; one rounding for *bound, one for +offset — same as the numpy generator
    dst[i] = __fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(u, 2.0f), 1.0f), bound), offset);
  }
}
void synth_fill_launch(float* dst, long long count, uint32_t key, float bound, float offset, cudaStream_t st) {
  int grid = (int)((count + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  synth_fill_kernel<<<grid, 256, 0, st>>>(dst, count, key, bound, offset);
  SDB_CUDA(cudaGetLastError());
}

// every tensor of the registry in ONE launch: a block walks 64K-element chunks; chunk -> tensor by binary search over the
// chunk prefix sums (one launch per tensor — 1131 of them — used to drown every other kernel in a profiler's launch list)
__global__ void __launch_bounds__(256)
synth_fill_table_kernel(float* __restrict__ base, const SynthDesc* __restrict__ desc, int ntensors, long long nchunks) {
  constexpr long long CH = 65536;
  for (long long ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    int lo = 0, hi = ntensors - 1;
    while (lo < hi) {  // last tensor whose first chunk is <= ch
      const int mid = (lo + hi + 1) >> 1;
      if (desc[mid].chunk0 <= ch) lo = mid; else hi = mid - 1;
    }
    const SynthDesc d = desc[lo];
    const long long i0 = (ch - d.chunk0) * CH, i1 = min(d.count, i0 + CH);
    float* dst = base + d.offset;
    for (long long i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
      const uint32_t h = mix32((uint32_t)i ^ d.key);
      const float u = (float)(h >> 8) * (1.0f / 16777216.0f);
      dst[i] = __fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(u, 2.0f), 1.0f), d.bound), d.shift);
    }
  }
}
void synth_fill_table_launch(float* base, const SynthDesc* d_desc, int ntensors, long long nchunks, cudaStream_t st) {
  const int grid = (int)std::min<long long>(nchunks, 148 * 16);
  synth_fill_table_kernel<<<grid, 256, 0, st>>>(base, d_desc, ntensors, nchunks);
  SDB_CUDA(cudaGetLastError());
}

}  // namespace sdb
