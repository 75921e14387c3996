// CUDA-core (fp32 FMA) implicit-GEMM multigrid convolution: forward, dgrad, wgrad.
//
// This is the "fp32 mode" of the hot path (north_star: rel 1e-4 against the oracle) and the
// on-device cross-check for the tcgen05 kernels in umma_conv.cu.  The cross-scale gather
// (2x2 max-pool of the finer grid | same grid | nearest-upsampled coarser grid, each with its
// producer's pending BatchNorm(+ReLU)) is evaluated on the fly inside the operand loader; the
// concatenated tensor of ResampleConcat (models/ilsvrc/rnmg.lua:41-89) never exists in HBM.
#include "common.cuh"
#include "conv_view.cuh"
#include <algorithm>

int simt_dbias(mg_ctx* ctx, const mg_grid* g, int Cout, float* dbias, float gscale);

namespace {

constexpr int TM = 64, TN = 64, TK = 16, NT = 256;

// C[i][j] = sum_l A(i,l) * B(l,j); blockIdx.z selects a slice of the reduction range.
template <class Prob>
__global__ void __launch_bounds__(NT) simt_gemm_kernel(Prob p) {
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const int i0 = blockIdx.x * TM, j0 = blockIdx.y * TN;
  const int64_t Ltot = p.L();
  const int64_t lper = (Ltot + gridDim.z - 1) / gridDim.z;
  const int64_t lbeg = blockIdx.z * lper;
  const int64_t lend = min(Ltot, lbeg + lper);

  // loader mapping: each thread owns one row (A) / one column (B) and 4 consecutive l
  const int la_i = tid / 4, la_l = (tid % 4) * 4;
  const int lb_j = tid / 4, lb_l = (tid % 4) * 4;
  auto actx = p.prepA(i0 + la_i);
  auto bctx = p.prepB(j0 + lb_j);

  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;

  for (int64_t l0 = lbeg; l0 < lend; l0 += TK) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int64_t l = l0 + la_l + q;
      As[la_l + q][la_i] = (l < lend) ? p.loadA(actx, l) : 0.f;
      l = l0 + lb_l + q;
      Bs[lb_l + q][lb_j] = (l < lend) ? p.loadB(bctx, l) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int l = 0; l < TK; ++l) {
      float a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[q] = As[l][ty * 4 + q]; b[q] = Bs[l][tx * 4 + q]; }
#pragma unroll
      for (int qa = 0; qa < 4; ++qa)
#pragma unroll
        for (int qb = 0; qb < 4; ++qb) acc[qa][qb] = fmaf(a[qa], b[qb], acc[qa][qb]);
    }
    __syncthreads();
  }
  p.epilogue(acc, i0 + ty * 4, j0 + tx * 4, tx, ty);
}

// ---------------------------------------------------------------- forward ------------
template <typename T>
struct FwdProb {
  ConvV<T> cv;
  const float* w;     // [Cout][Ccat][k][k]
  const float* bias;  // [Cout] or null
  T* y;               // [M][Cp_out]
  int y_cp;
  mg_sum* bn_sums;    // [2*Cout] or null
  int64_t M;
  __device__ int64_t L() const { return (int64_t)cv.k * cv.k * cv.Ccat; }
  struct ACtx { int n, oy, ox; bool valid; };
  __device__ ACtx prepA(int64_t m) const {
    ACtx c; c.valid = m < M;
    int64_t mm = c.valid ? m : 0;
    c.ox = mm % cv.Wo; mm /= cv.Wo; c.oy = mm % cv.Ho; c.n = mm / cv.Ho;
    return c;
  }
  __device__ float loadA(const ACtx& c, int64_t l) const {
    if (!c.valid) return 0.f;
    int tap = l / cv.Ccat, ci = l % cv.Ccat;
    int ky = tap / cv.k, kx = tap % cv.k;
    int iy = c.oy * cv.stride + ky - cv.pad, ix = c.ox * cv.stride + kx - cv.pad;
    if (iy < 0 || iy >= cv.H || ix < 0 || ix >= cv.W) return 0.f;
    return cv.fetch(c.n, iy, ix, ci);
  }
  struct BCtx { int co; };
  __device__ BCtx prepB(int64_t j) const { return BCtx{(int)j}; }
  __device__ float loadB(const BCtx& c, int64_t l) const {
    if (c.co >= cv.Cout) return 0.f;
    int tap = l / cv.Ccat, ci = l % cv.Ccat;
    return w[((size_t)c.co * cv.Ccat + ci) * cv.k * cv.k + tap];
  }
  __device__ void epilogue(float (&acc)[4][4], int64_t m0, int co0, int tx, int ty) const {
    // per-thread partial sums staged by tile row (ty) and added in a fixed order: no floating-point atomics, the CTA's
    // contribution is the same from run to run; across CTAs the totals are deterministic integer sums (mg_sum)
    __shared__ float red[2][TM / 4][TN];
#pragma unroll
    for (int qb = 0; qb < 4; ++qb) {
      int co = co0 + qb;
      float s = 0.f, s2 = 0.f;
      if (co < cv.Cout) {
        float b = bias ? bias[co] : 0.f;
#pragma unroll
        for (int qa = 0; qa < 4; ++qa) {
          int64_t m = m0 + qa;
          if (m < M) {
            float v = acc[qa][qb] + b;
            mg_st(y + m * y_cp + co, v);
            s += v; s2 += v * v;
          }
        }
      }
      if (bn_sums) { red[0][ty][tx * 4 + qb] = s; red[1][ty][tx * 4 + qb] = s2; }
    }
    if (bn_sums) {
      __syncthreads();
      int t = threadIdx.x;
      if (t < TN) {
        int co = blockIdx.y * TN + t;
        if (co < cv.Cout) {
          float a = 0.f, b2 = 0.f;
          for (int r = 0; r < TM / 4; ++r) { a += red[0][r][t]; b2 += red[1][r][t]; }
          mg_sum_add(bn_sums + co, (double)a);
          mg_sum_add(bn_sums + cv.Cout + co, (double)b2);
        }
      }
    }
  }
};

// ---------------------------------------------------------------- dgrad --------------
// dcat[m][cpad] = sum_{ky,kx,co} g[n, y+pad-ky, x+pad-kx, co] * w[co][ci][ky][kx]   (stride 1)
template <typename T>
struct DgradProb {
  ConvV<T> cv;
  const float* w;
  const T* g;  // [M][g_cp]
  int g_cp;
  T* dcat;     // [M][CcatP]
  int64_t M;
  __device__ int64_t L() const { return (int64_t)cv.k * cv.k * cv.Cout; }
  struct ACtx { int n, y, x; bool valid; };
  __device__ ACtx prepA(int64_t m) const {
    ACtx c; c.valid = m < M;
    int64_t mm = c.valid ? m : 0;
    c.x = mm % cv.W; mm /= cv.W; c.y = mm % cv.H; c.n = mm / cv.H;
    return c;
  }
  __device__ float loadA(const ACtx& c, int64_t l) const {
    if (!c.valid) return 0.f;
    int tap = l / cv.Cout, co = l % cv.Cout;
    int ky = tap / cv.k, kx = tap % cv.k;
    int oy = c.y + cv.pad - ky, ox = c.x + cv.pad - kx;
    if (oy < 0 || oy >= cv.Ho || ox < 0 || ox >= cv.Wo) return 0.f;
    return mg_ld(g + (((size_t)c.n * cv.Ho + oy) * cv.Wo + ox) * g_cp + co);
  }
  struct BCtx { int ci; };  // logical concat channel or -1 for a pad channel
  __device__ BCtx prepB(int64_t j) const { return BCtx{cv.logical_of_padded((int)j)}; }
  __device__ float loadB(const BCtx& c, int64_t l) const {
    if (c.ci < 0) return 0.f;
    int tap = l / cv.Cout, co = l % cv.Cout;
    return w[((size_t)co * cv.Ccat + c.ci) * cv.k * cv.k + tap];
  }
  __device__ void epilogue(float (&acc)[4][4], int64_t m0, int c0, int, int) const {
#pragma unroll
    for (int qa = 0; qa < 4; ++qa) {
      int64_t m = m0 + qa;
      if (m >= M) continue;
#pragma unroll
      for (int qb = 0; qb < 4; ++qb)
        if (c0 + qb < cv.CcatP) mg_st(dcat + m * cv.CcatP + c0 + qb, acc[qa][qb]);
    }
  }
};

// ---------------------------------------------------------------- wgrad --------------
// dw[co][ci][ky][kx] += gscale * sum_m g[m][co] * gather(m, ky, kx, ci)
template <typename T>
struct WgradProb {
  ConvV<T> cv;
  const T* g;
  int g_cp;
  float* partial;   // [splits][Cout][k*k*Ccat] partial sums (context workspace); simt_wgrad_reduce_kernel adds them in a fixed order
  int64_t M;
  __device__ int64_t L() const { return M; }
  struct ACtx { int co; };
  __device__ ACtx prepA(int64_t i) const { return ACtx{(int)i}; }
  __device__ float loadA(const ACtx& c, int64_t m) const {
    if (c.co >= cv.Cout) return 0.f;
    return mg_ld(g + (size_t)m * g_cp + c.co);
  }
  struct BCtx { int ky, kx, ci; bool valid; };
  __device__ BCtx prepB(int64_t j) const {
    BCtx c; c.valid = j < (int64_t)cv.k * cv.k * cv.Ccat;
    int jj = c.valid ? (int)j : 0;
    int tap = jj / cv.Ccat; c.ci = jj % cv.Ccat; c.ky = tap / cv.k; c.kx = tap % cv.k;
    return c;
  }
  __device__ float loadB(const BCtx& c, int64_t m) const {
    if (!c.valid) return 0.f;
    int64_t mm = m;
    int ox = mm % cv.Wo; mm /= cv.Wo; int oy = mm % cv.Ho; int n = mm / cv.Ho;
    int iy = oy * cv.stride + c.ky - cv.pad, ix = ox * cv.stride + c.kx - cv.pad;
    if (iy < 0 || iy >= cv.H || ix < 0 || ix >= cv.W) return 0.f;
    return cv.fetch(n, iy, ix, c.ci);
  }
  __device__ void epilogue(float (&acc)[4][4], int64_t co0, int j0, int, int) const {
    const int KK = cv.k * cv.k;
#pragma unroll
    for (int qa = 0; qa < 4; ++qa) {
      int co = co0 + qa;
      if (co >= cv.Cout) continue;
#pragma unroll
      for (int qb = 0; qb < 4; ++qb) {
        int j = j0 + qb;
        if (j >= KK * cv.Ccat) continue;
        partial[((size_t)blockIdx.z * cv.Cout + co) * ((size_t)KK * cv.Ccat) + j] = acc[qa][qb];
      }
    }
  }
};

// dw[co][ci][tap] += gscale * sum_z partial[z][co][tap * Ccat + ci]   (z in increasing order: no floating-point atomics)
__global__ void simt_wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int Cout, int Ccat, int KK, float* __restrict__ dw, float gscale) {
  const int64_t plane = (int64_t)Cout * KK * Ccat;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += partial[(size_t)z * plane + i];
  const int j = (int)(i % ((int64_t)KK * Ccat)), co = (int)(i / ((int64_t)KK * Ccat));
  const int tap = j / Ccat, ci = j % Ccat;
  dw[((size_t)co * Ccat + ci) * KK + tap] += gscale * s;
}

// scratch[c] += sum_m g[m][c] (deterministic integer accumulation across blocks), then dbias_finalize_kernel:
// dbias[c] += gscale * scratch[c]; scratch[c] = 0
template <typename T>
__global__ void dbias_kernel(const T* g, int cp, int C, int64_t M, mg_sum* scratch) {
  int c = blockIdx.x * 32 + (threadIdx.x % 32);
  int lane_row = threadIdx.x / 32;
  int rows_per_block = blockDim.x / 32;
  float s = 0.f;
  if (c < C)
    for (int64_t m = (int64_t)blockIdx.y * rows_per_block + lane_row; m < M; m += (int64_t)gridDim.y * rows_per_block)
      s += mg_ld(g + m * cp + c);
  __shared__ float red[8][33];
  red[lane_row][threadIdx.x % 32] = s;
  __syncthreads();
  if (lane_row == 0 && c < C) {
    float t = 0.f;
    for (int r = 0; r < rows_per_block; ++r) t += red[r][threadIdx.x % 32];
    mg_sum_add(scratch + c, (double)t);
  }
}

__global__ void dbias_finalize_kernel(mg_sum* scratch, int C, float* dbias, float gscale) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  dbias[c] += gscale * (float)mg_sum_get(scratch[c]);
  scratch[c].hi = 0; scratch[c].lo = 0;
}

}  // namespace

template <typename T>
static int simt_forward_t(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const float* bias,
                          mg_grid* y, mg_sum* bn_sums) {
  FwdProb<T> p;
  int rc = make_conv_view<T>(ctx, *d, &p.cv);
  if (rc) return rc;
  p.w = w; p.bias = bias; p.y = (T*)y->data; p.y_cp = y->Cp; p.bn_sums = bn_sums;
  p.M = (int64_t)p.cv.N * p.cv.Ho * p.cv.Wo;
  dim3 grid((unsigned)mg_cdiv(p.M, TM), (unsigned)mg_cdiv(d->Cout, TN), 1);
  simt_gemm_kernel<<<grid, NT, 0, ctx->stream>>>(p);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int simt_conv_forward(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const float* bias,
                      mg_grid* y, mg_sum* bn_sums) {
  MG_DISPATCH(ctx, return simt_forward_t<T>(ctx, d, w, bias, y, bn_sums););
}

template <typename T>
static int simt_dgrad_t(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const mg_grid* g, mg_grid* dcat) {
  DgradProb<T> p;
  int rc = make_conv_view<T>(ctx, *d, &p.cv);
  if (rc) return rc;
  MG_REQUIRE(ctx, d->stride == 1, MG_ERR_UNSUPPORTED, "dgrad: stride %d goes through simt_strided_dgrad", d->stride);
  p.w = w; p.g = (const T*)g->data; p.g_cp = g->Cp; p.dcat = (T*)dcat->data;
  p.M = (int64_t)p.cv.N * p.cv.H * p.cv.W;
  MG_REQUIRE(ctx, dcat->Cp == p.cv.CcatP, MG_ERR_SHAPE, "dgrad: dcat.Cp %d != %d", dcat->Cp, p.cv.CcatP);
  dim3 grid((unsigned)mg_cdiv(p.M, TM), (unsigned)mg_cdiv(p.cv.CcatP, TN), 1);
  simt_gemm_kernel<<<grid, NT, 0, ctx->stream>>>(p);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int simt_conv_backward_data(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const mg_grid* g, mg_grid* dcat) {
  MG_DISPATCH(ctx, return simt_dgrad_t<T>(ctx, d, w, g, dcat););
}

// Data gradient of the image-fed strided stem, cudnn.SpatialConvolution(3, C, 7,7, 2,2, 3,3) (models/ilsvrc/rnmg.lua:180):
//   dx[n][iy][ix][ci] = sum over (ky, kx) with iy = oy*stride - pad + ky, ix = ox*stride - pad + kx, and over co, of
//                       g[n][oy][ox][co] * w[co][ci][ky][kx].
// A CUDA-core kernel, not a tcgen05 one: the output has 3 channels (one 8-channel vector), far below the N >= 16 of an MMA, while
// the reduction (49 taps x Cout) is long.  The whole fp32 weight tensor sits in shared memory as [ky][kx][co][ci]; one thread owns
// one input pixel, visits only the taps of its parity class ((iy + pad - ky) divisible by the stride: 16 of 49 for 7x7 / 2) and
// accumulates its <= 8 channels in registers in a fixed order, so the result is deterministic.
template <typename T>
__global__ void __launch_bounds__(128) stem_dgrad_kernel(const T* __restrict__ g, int g_cp, int Ho, int Wo, int Cout, const float* __restrict__ w,
                                                         int Cin, int k, int stride, int pad, T* __restrict__ dx, int dx_cp, int N, int H, int W) {
  extern __shared__ float s_w[];
  const int taps = k * k;
  for (int i = threadIdx.x; i < taps * Cout * Cin; i += blockDim.x) {
    const int ci = i % Cin, r = i / Cin, co = r % Cout, t = r / Cout;
    s_w[i] = w[((size_t)co * Cin + ci) * taps + t];
  }
  __syncthreads();
  const int64_t P = (int64_t)N * H * W;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < P; pix += (int64_t)gridDim.x * blockDim.x) {
    const int ix = (int)(pix % W);
    const int64_t q = pix / W;
    const int iy = (int)(q % H), n = (int)(q / H);
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    for (int ky = (iy + pad) % stride; ky < k; ky += stride) {
      const int oy = (iy + pad - ky) / stride;   // exact: iy + pad - ky is a multiple of the stride
      if (iy + pad - ky < 0 || oy >= Ho) continue;
      for (int kx = (ix + pad) % stride; kx < k; kx += stride) {
        const int ox = (ix + pad - kx) / stride;
        if (ix + pad - kx < 0 || ox >= Wo) continue;
        const T* gp = g + (((size_t)n * Ho + oy) * Wo + ox) * g_cp;
        const float* wp = s_w + (size_t)(ky * k + kx) * Cout * Cin;
        for (int co = 0; co < Cout; ++co) {
          const float gv = mg_ld(gp + co);
#pragma unroll
          for (int ci = 0; ci < 8; ++ci)
            if (ci < Cin) acc[ci] = fmaf(gv, wp[co * Cin + ci], acc[ci]);
        }
      }
    }
    T* o = dx + pix * dx_cp;
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (c < dx_cp) mg_st(o + c, c < Cin ? acc[c] : 0.f);
  }
}

template <typename T>
static int stem_dgrad_t(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const mg_grid* g, mg_grid* dcat) {
  const mg_grid& x = d->seg[0];
  MG_REQUIRE(ctx, d->n_seg == 1 && d->seg_mode[0] == MG_SEG_SAME && !x.scale && x.C <= 8 && x.Cp == 8 && dcat->Cp == 8, MG_ERR_UNSUPPORTED,
             "dgrad: a strided convolution needs one unresampled input of at most 8 channels (the image-fed stem)");
  const int Ho = (d->H + 2 * d->pad - d->ksize) / d->stride + 1, Wo = (d->W + 2 * d->pad - d->ksize) / d->stride + 1;
  MG_REQUIRE(ctx, g->H == Ho && g->W == Wo && g->N == x.N && dcat->N == x.N, MG_ERR_SHAPE, "dgrad: g is %dx%d, expected %dx%d", g->H, g->W, Ho, Wo);
  const size_t smem = (size_t)d->ksize * d->ksize * d->Cout * x.C * sizeof(float);
  MG_REQUIRE(ctx, smem <= 200 * 1024, MG_ERR_UNSUPPORTED, "dgrad: strided weights of %zu bytes exceed shared memory", smem);
  if (smem > 48 * 1024)
    MG_CUDA(ctx, cudaFuncSetAttribute(stem_dgrad_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t P = (int64_t)x.N * d->H * d->W;
  const unsigned grid = (unsigned)std::min<int64_t>(mg_cdiv(P, (int64_t)128), (int64_t)ctx->num_sms * 8);
  stem_dgrad_kernel<T><<<grid, 128, smem, ctx->stream>>>((const T*)g->data, g->Cp, Ho, Wo, d->Cout, w, x.C, d->ksize, d->stride, d->pad,
                                                         (T*)dcat->data, dcat->Cp, x.N, d->H, d->W);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int simt_strided_dgrad(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const mg_grid* g, mg_grid* dcat) {
  MG_DISPATCH(ctx, return stem_dgrad_t<T>(ctx, d, w, g, dcat););
}

template <typename T>
static int simt_wgrad_t(mg_ctx* ctx, const mg_conv_desc* d, const mg_grid* g, float* dw, float* dbias, float gscale) {
  WgradProb<T> p;
  int rc = make_conv_view<T>(ctx, *d, &p.cv);
  if (rc) return rc;
  p.g = (const T*)g->data; p.g_cp = g->Cp;
  p.M = (int64_t)p.cv.N * p.cv.Ho * p.cv.Wo;
  int KK = d->ksize * d->ksize * p.cv.Ccat;
  int gx = (int)mg_cdiv(d->Cout, TM), gy = (int)mg_cdiv(KK, TN);
  // split the pixel reduction so that the grid covers the machine a few times
  int64_t want = (int64_t)ctx->num_sms * 4;
  int gz = (int)std::max<int64_t>(1, std::min<int64_t>(mg_cdiv(want, (int64_t)gx * gy), mg_cdiv(p.M, 256)));
  dim3 grid(gx, gy, gz);
  const int64_t plane = (int64_t)d->Cout * KK;
  void* ws = nullptr;
  rc = mg_ctx_workspace(ctx, (size_t)gz * plane * sizeof(float), &ws);
  if (rc) return rc;
  p.partial = (float*)ws;
  simt_gemm_kernel<<<grid, NT, 0, ctx->stream>>>(p);
  MG_CHECK_LAUNCH(ctx);
  simt_wgrad_reduce_kernel<<<(unsigned)mg_cdiv(plane, 256), 256, 0, ctx->stream>>>(p.partial, gz, d->Cout, p.cv.Ccat, d->ksize * d->ksize, dw, gscale);
  MG_CHECK_LAUNCH(ctx);
  if (dbias) return simt_dbias(ctx, g, d->Cout, dbias, gscale);
  return MG_OK;
}

template <typename T>
static int simt_dbias_t(mg_ctx* ctx, const mg_grid* g, int Cout, float* dbias, float gscale) {
  const int64_t M = (int64_t)g->N * g->H * g->W;
  MG_REQUIRE(ctx, Cout <= MG_SUM_SCRATCH, MG_ERR_UNSUPPORTED, "dbias: %d channels", Cout);
  mg_sum* scratch = mg_ctx_sum_scratch(ctx);
  MG_REQUIRE(ctx, scratch != nullptr, MG_ERR_CUDA, "dbias: scratch allocation failed");
  dim3 g2((unsigned)mg_cdiv(Cout, 32), (unsigned)std::min<int64_t>(mg_cdiv(M, 64), 256));
  dbias_kernel<T><<<g2, 256, 0, ctx->stream>>>((const T*)g->data, g->Cp, Cout, M, scratch);
  MG_CHECK_LAUNCH(ctx);
  dbias_finalize_kernel<<<(unsigned)mg_cdiv(Cout, 256), 256, 0, ctx->stream>>>(scratch, Cout, dbias, gscale);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// dbias += gscale * sum over pixels of g (accGradParameters' gradBias)
int simt_dbias(mg_ctx* ctx, const mg_grid* g, int Cout, float* dbias, float gscale) {
  MG_DISPATCH(ctx, return simt_dbias_t<T>(ctx, g, Cout, dbias, gscale););
}

int simt_conv_backward_weight(mg_ctx* ctx, const mg_conv_desc* d, const mg_grid* g, float* dw, float* dbias, float gscale) {
  MG_DISPATCH(ctx, return simt_wgrad_t<T>(ctx, d, g, dw, dbias, gscale););
}
