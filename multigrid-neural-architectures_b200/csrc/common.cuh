// Shared device/host helpers of libmgconv (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <curand_philox4x32_x.h>
#include "../../include/mgconv.h"

#define MG_MAX_LANES 4
#define MG_SUM_SCRATCH 4096
struct mg_ctx {
  int device;
  cudaStream_t stream;      // stream every call enqueues on = lane_stream[cur_lane]
  int dtype;        // mg_dtype
  int impl;         // mg_impl
  int num_sms;
  int64_t launches; // kernels launched through this context
  int64_t tc_launches; // of which tcgen05 (UMMA) kernels
  char err[512];
  // data parallel
  void* nccl_comm;
  cudaStream_t comm_stream;
  cudaEvent_t ev_compute, ev_comm;
  int rank, nranks;
  int comm_borrowed;   // mg_comm_share: nccl_comm belongs to another context (never destroyed here)
  // optional CUDA-event timing of the convolution kernels (bench.py roofline)
  int profile;
  void* prof;  // ProfState*
  // scratch owned by the context (split-K partial sums of the weight gradient), grown on demand
  void* ws;
  size_t ws_bytes;
  // lanes (mg_ctx_lane): lane 0 is the caller's stream, lanes 1.. are side streams owned by the context; each lane
  // has its own scratch, so independent chains of a stage (one per scale) may run concurrently
  cudaStream_t lane_stream[MG_MAX_LANES];
  int cur_lane;
  void* lane_ws[MG_MAX_LANES];        // scratch of lanes 1.. (lane 0 uses ws)
  size_t lane_ws_bytes[MG_MAX_LANES];
  void* up_ws[MG_MAX_LANES];          // scratch of the tensor-core up-convolution (upconv_tc.cu), per lane
  size_t up_ws_bytes[MG_MAX_LANES];
  cudaEvent_t* events;                // mg_ctx_event_record / mg_ctx_event_wait pool
  int n_events;
  cudaEvent_t lane_ev[MG_MAX_LANES];  // mg_allreduce_launch: completion of everything enqueued so far on each lane
  // kernel-selection overrides (mg_ctx_set_tuning); 0 = automatic
  int tune_mt;       // 128-slot sub-tiles per CTA of the halo convolution kernel (1 / 2)
  int tune_persist;  // weight-resident persistent kernel: 1 = whenever the weights fit, 2 = never
  int tune_stem_fused;  // stem kernel: 1 = BatchNorm sums in its epilogue, 0 = separate statistics pass (faster, default)
  // job table of mg_conv_pack_weights_batched (device copy + the host image it was uploaded from)
  mg_sum* sum_scratch[MG_MAX_LANES];   // zeroed scratch of MG_SUM_SCRATCH deterministic sums per lane (users re-zero what they used)
  void* tmaps;         // TmapCache* (tma.cuh): CUtensorMap objects of the halo kernels, keyed by (pointer, shape)
  void* pack_dev;
  void* pack_host;
  size_t pack_cap, pack_bytes;
};

// make the context workspace at least `bytes` large (one blocking cudaMalloc when it grows)
static inline int mg_ctx_workspace(mg_ctx* ctx, size_t bytes, void** out) {
  void** ws = ctx->cur_lane ? &ctx->lane_ws[ctx->cur_lane] : &ctx->ws;
  size_t* cap = ctx->cur_lane ? &ctx->lane_ws_bytes[ctx->cur_lane] : &ctx->ws_bytes;
  if (*cap < bytes) {
    if (*ws) { cudaStreamSynchronize(ctx->stream); cudaFree(*ws); *ws = nullptr; *cap = 0; }
    if (cudaMalloc(ws, bytes) != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "workspace: cudaMalloc(%zu) failed", bytes); return MG_ERR_CUDA; }
    *cap = bytes;
  }
  *out = *ws;
  return MG_OK;
}

// zeroed per-lane scratch of deterministic sums; a user must leave it zeroed (its finalising kernel re-zeroes what it read)
static inline mg_sum* mg_ctx_sum_scratch(mg_ctx* ctx) {
  mg_sum** s = &ctx->sum_scratch[ctx->cur_lane];
  if (!*s) {
    if (cudaMalloc((void**)s, MG_SUM_SCRATCH * sizeof(mg_sum)) != cudaSuccess) { *s = nullptr; return nullptr; }
    cudaMemsetAsync(*s, 0, MG_SUM_SCRATCH * sizeof(mg_sum), ctx->stream);
  }
  return *s;
}

#define MG_FAIL(ctx, code, ...)                                  \
  do {                                                           \
    if (ctx) snprintf((ctx)->err, sizeof((ctx)->err), __VA_ARGS__); \
    return (code);                                               \
  } while (0)

#define MG_CUDA(ctx, expr)                                                        \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess)                                                        \
      MG_FAIL(ctx, MG_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
  } while (0)

#define MG_CHECK_LAUNCH(ctx)              \
  do {                                    \
    (ctx)->launches++;                    \
    MG_CUDA(ctx, cudaGetLastError());     \
  } while (0)

#define MG_REQUIRE(ctx, cond, code, ...) \
  do {                                   \
    if (!(cond)) MG_FAIL(ctx, code, __VA_ARGS__); \
  } while (0)

static inline int mg_round_up(int a, int b) { return (a + b - 1) / b * b; }
static inline int64_t mg_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- element access --------------------------------------------------------------
__device__ __forceinline__ float mg_ld(const float* p) { return *p; }
__device__ __forceinline__ float mg_ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void mg_st(float* p, float v) { *p = v; }
__device__ __forceinline__ void mg_st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// pending affine (+ReLU) of a grid; identical expression everywhere so that forward
// values, ReLU masks and pool arg-maxima agree bit for bit between kernels
__device__ __forceinline__ float mg_xform(float v, float sc, float sh, int relu) {
  float a = fmaf(v, sc, sh);
  return relu ? fmaxf(a, 0.f) : a;
}

// device view of a grid
template <typename T>
struct GridV {
  const T* data;
  const float* scale;
  const float* shift;
  int relu;
  int N, H, W, C, Cp;
  __device__ __forceinline__ float raw(int n, int y, int x, int c) const {
    return mg_ld(data + (((size_t)n * H + y) * W + x) * Cp + c);
  }
  __device__ __forceinline__ float at(int n, int y, int x, int c) const {
    float v = raw(n, y, x, c);
    if (scale) v = mg_xform(v, scale[c], shift[c], relu);
    return v;
  }
  // SpatialMaxPooling(2,2,2,2,0,0):ceil() window at pooled position (py,px): rows then cols,
  // strict '>' so the first maximum wins; *arg = flat y*W+x of the winner
  __device__ __forceinline__ float pooled(int n, int py, int px, int c, int* arg) const {
    int y0 = 2 * py, x0 = 2 * px;
    int y1 = min(y0 + 2, H), x1 = min(x0 + 2, W);
    float best = -INFINITY;
    int bi = y0 * W + x0;
    for (int yy = y0; yy < y1; ++yy)
      for (int xx = x0; xx < x1; ++xx) {
        float v = at(n, yy, xx, c);
        if (v > best || v != v) { best = v; bi = yy * W + xx; }
      }
    if (arg) *arg = bi;
    return best;
  }
};

template <typename T>
static inline GridV<T> make_view(const mg_grid& g) {
  GridV<T> v;
  v.data = (const T*)g.data; v.scale = g.scale; v.shift = g.shift; v.relu = g.relu;
  v.N = g.N; v.H = g.H; v.W = g.W; v.C = g.C; v.Cp = g.Cp;
  return v;
}

static inline size_t mg_elt_size(int dtype) { return dtype == MG_BF16 ? 2 : 4; }

// ---- counter-based dropout mask (mg_dropout, see mgconv.h) ------------------------------------------------------
// element i (NHWC index over the logical channels) is kept iff word i & 3 of Philox4x32-10((i >> 2, op, step, rank), seed) >= t
struct DropK {
  uint32_t key_lo, key_hi, op, rank, t;
  float s;                 // fp32(1 / (1 - p))
  const uint64_t* step;
};

// bit e of the result: element i0 + e is kept (n <= 8 consecutive elements, at most three Philox calls)
__device__ __forceinline__ uint32_t drop_keep_bits(uint64_t i0, int n, const DropK& k) {
  const uint32_t step = (uint32_t)*k.step;
  uint32_t bits = 0;
  for (uint64_t g = i0 >> 2; g <= (i0 + n - 1) >> 2; ++g) {
    const uint4 u = curand_Philox4x32_10(make_uint4((uint32_t)g, k.op, step, k.rank), make_uint2(k.key_lo, k.key_hi));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t e = (int64_t)(4 * g + j) - (int64_t)i0;
      if (e >= 0 && e < n && w[j] >= k.t) bits |= 1u << e;
    }
  }
  return bits;
}

// the source segments of mg_dropout_forward: output channel c belongs to segment s when off[s] <= c < off[s + 1]
template <typename T>
struct DropSegs {
  int n;
  GridV<T> g[MG_MAX_SEG];
  int up[MG_MAX_SEG];      // MG_SEG_UP: read at (y / 2, x / 2)
  int off[MG_MAX_SEG + 1];
};
template <typename T>
static inline DropSegs<T> make_drop_segs(int n, const mg_grid* seg, const int32_t* mode) {
  DropSegs<T> d;
  memset(&d, 0, sizeof(d));
  d.n = n;
  for (int s = 0; s < n; ++s) {
    d.g[s] = make_view<T>(seg[s]);
    d.up[s] = mode[s] == MG_SEG_UP;
    d.off[s + 1] = d.off[s] + seg[s].C;
  }
  return d;
}
// value of output channel c at (n, y, x) of the concatenation
template <typename T>
__device__ __forceinline__ float drop_gather(const DropSegs<T>& d, int n, int y, int x, int c) {
  int s = 0;
  while (s + 1 < d.n && c >= d.off[s + 1]) ++s;
  return d.up[s] ? d.g[s].at(n, y >> 1, x >> 1, c - d.off[s]) : d.g[s].at(n, y, x, c - d.off[s]);
}

// dispatch on the context dtype
#define MG_DISPATCH(ctx, ...)                          \
  do {                                                 \
    if ((ctx)->dtype == MG_BF16) { using T = __nv_bfloat16; __VA_ARGS__ } \
    else { using T = float; __VA_ARGS__ }              \
  } while (0)

// block-wide helpers
__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- deterministic sums (mg_sum, see mgconv.h): value = hi * 2^-10 + lo * 2^-54 ------------------------------
__device__ __forceinline__ void mg_to_fix(double v, long long& hi, long long& lo) {
  const double s = v * 1024.0;
  if (fabs(s) < 1.0e15) {
    const double f = floor(s);
    hi = (long long)f;
    lo = (long long)((s - f) * 17592186044416.0);   // 2^44; truncation: a deterministic function of v
  } else {   // out of range / inf / nan: poison the sum (read back as NaN)
    hi = 1ll << 61; lo = 0;
  }
}
// the same conversion for an fp32 value without fp64 instructions: v * 2^10, its floor, the remainder and its scaling by 2^44 are
// all exact in fp32 (power-of-two scalings; the remainder of a 24-bit number has at most 24 bits), so the result is bit-identical
// to mg_to_fix((double)v)
__device__ __forceinline__ void mg_to_fix_f32(float v, long long& hi, long long& lo) {
  const float s = v * 1024.0f;
  if (fabsf(s) < 1.0e15f) {
    const float f = floorf(s);
    hi = __float2ll_rz(f);
    lo = __float2ll_rz((s - f) * 17592186044416.0f);
  } else {
    hi = 1ll << 61; lo = 0;
  }
}
__device__ __forceinline__ void mg_sum_add_fix(mg_sum* p, long long hi, long long lo) {
  atomicAdd(reinterpret_cast<unsigned long long*>(&p->hi), (unsigned long long)hi);
  atomicAdd(reinterpret_cast<unsigned long long*>(&p->lo), (unsigned long long)lo);
}
__device__ __forceinline__ void mg_sum_add(mg_sum* p, double v) {
  long long hi, lo;
  mg_to_fix(v, hi, lo);
  mg_sum_add_fix(p, hi, lo);
}
__host__ __device__ __forceinline__ double mg_sum_get(const mg_sum& s) {
  if (s.hi >= (1ll << 60) || s.hi <= -(1ll << 60)) return nan("");
  return (double)s.hi * (1.0 / 1024.0) + (double)s.lo * (1.0 / 18014398509481984.0);   // 2^-54
}

// BatchNorm in evaluation mode ("frozen": running statistics, no update): invstd_r = 1 / sqrt(running_var + eps) in fp64, the
// expression of mg_bn_finalize.  FrozenBn carries what mg_grad_combine_bn_frozen hands to the combine kernels.
__device__ __forceinline__ double frozen_bn_invstd(float rvar, float eps) { return 1.0 / sqrt((double)rvar + (double)eps); }
struct FrozenBn { const float* gamma; const float* running_var; float eps; const mg_grid* g; };

// Training-mode BatchNorm backward of one channel from the sums sd = sum d, sdx = sum d*y over n elements, the batch mean mu,
// invstd `is` and gamma g: dg = is * (sdx - mu * sd) and the coefficients of G = A*d + B*y + C.  RECIP divides by n through
// rn = 1 / n (the one-pass bf16 kernel: no fp64 division per CTA), else by n itself (the fp32 coefficient kernel).  Every
// kernel that derives these terms (mg_bn_backward, mg_bn_backward_frozen, mg_bn_param_grad) goes through the functions below,
// written operation by operation with the _rn intrinsics, which the compiler never contracts or reorders: the rounding of each
// step is fixed by the source, not by how the surrounding kernel was scheduled, so the split backward adds exactly the bits of
// the fused one.  (The steps are the ones nvcc made of the plain expressions these functions replace.)
struct BnTrainTerms { double dg, Ad, Bd, Cd; };
template <bool RECIP>
__device__ __forceinline__ BnTrainTerms bn_train_terms(double sd, double sdx, double mu, double is, double g, double n, double rn) {
  BnTrainTerms t;
  t.dg = __dmul_rn(is, __fma_rn(mu, -sd, sdx));                  // is * (sdx - mu * sd)
  t.Ad = __dmul_rn(g, is);
  const double b = __dmul_rn(__dmul_rn(-t.Ad, is), t.dg);         // -g * is * is * dg
  const double x = __dmul_rn(__dmul_rn(mu, is), t.dg);            // mu * is * dg
  if (RECIP) {
    t.Bd = __dmul_rn(b, rn);
    t.Cd = __dmul_rn(t.Ad, __fma_rn(x, rn, -__dmul_rn(sd, rn)));  // g * is * (x / n - sd / n)
  } else {
    t.Bd = __ddiv_rn(b, n);
    t.Cd = __dmul_rn(t.Ad, __dsub_rn(__ddiv_rn(x, n), __ddiv_rn(sd, n)));
  }
  return t;
}
// dgamma += gscale * dg, dbeta += gscale * sum d, and the gradBias of the convolution that produced y += gscale * sum over
// pixels of G = A * sum d + B * sum y + C * n (identically zero in exact arithmetic: rounding noise in the reference as well)
__device__ __forceinline__ void bn_train_param_grad(const BnTrainTerms& t, double sd, double mu, double n, int c, float* dgamma,
                                                    float* dbeta, float* conv_dbias, float gscale) {
  if (dgamma) dgamma[c] = __fmaf_rn((float)t.dg, gscale, dgamma[c]);
  if (dbeta) dbeta[c] = __fmaf_rn((float)sd, gscale, dbeta[c]);
  if (conv_dbias) {
    const double s = __fma_rn(n, t.Cd, __fma_rn(t.Ad, sd, __dmul_rn(t.Bd, __dmul_rn(mu, n))));
    conv_dbias[c] = __fmaf_rn((float)s, gscale, conv_dbias[c]);
  }
}
// frozen BatchNorm: dgamma += gscale * invstd_r * (sum d*y - mu_r * sum d), dbeta += gscale * sum d and the producing
// convolution's gradBias += gscale * A * sum d (= the pixel sum of G = A * d), A = gamma * invstd_r
__device__ __forceinline__ void bn_frozen_param_grad(const mg_sum* sums, int C, int c, const float* gamma, const float* rmean,
                                                     const float* rvar, float eps, float* dgamma, float* dbeta, float gscale,
                                                     float* conv_dbias) {
  const double sd = mg_sum_get(sums[c]), sdy = mg_sum_get(sums[C + c]);
  const double is = frozen_bn_invstd(rvar[c], eps);
  if (dgamma) dgamma[c] = __fmaf_rn((float)__dmul_rn(is, __fma_rn((double)rmean[c], -sd, sdy)), gscale, dgamma[c]);
  if (dbeta) dbeta[c] = __fmaf_rn((float)sd, gscale, dbeta[c]);
  const float A = (float)__dmul_rn(gamma ? (double)gamma[c] : 1.0, is);
  if (conv_dbias) conv_dbias[c] = __fmaf_rn((float)__dmul_rn((double)A, sd), gscale, conv_dbias[c]);
}

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------
// A kernel launched with mg_launch_pdl may become resident while its predecessor in the stream is still
// draining; it must execute pdl_wait() before touching anything the predecessor wrote.  pdl_launch() (first
// statement of every such kernel) lets the NEXT kernel start its launch once all CTAs of this grid started.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

static inline bool mg_pdl_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("MGCONV_PDL"); on = e ? atoi(e) : 1; }
  return on != 0;
}

template <typename... KArgs, typename... Args>
static inline cudaError_t mg_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = mg_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
