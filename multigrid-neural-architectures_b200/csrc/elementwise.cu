// HBM-bound passes of the multigrid hot path: layout import/export, BatchNorm finalise and
// backward, residual add, pooling, the gradient "combine" (gather-form scatter through pool
// arg-max / upsample / shortcut), criteria and SGD.  One thread per (pixel, channel) with the
// channel index fastest, so a warp touches 32 consecutive channels of one NHWC pixel row.
#include "common.cuh"
#include <algorithm>

// bf16 fast paths (elementwise_bf16.cu); each returns false when it does not apply
bool bf16_im2col(mg_ctx*, const mg_grid* in, int k, int stride, int pad, mg_grid* col);
int upconv_tc_forward(mg_ctx*, const mg_grid* x, const float* w, const float* bias, mg_grid* y);
int upconv_tc_backward(mg_ctx*, const mg_grid* x, const float* w, const mg_grid* g, mg_grid* dx, float* dw, float* dbias, float gscale);
bool bf16_apply(mg_ctx*, const mg_grid* z, const mg_grid* s, int relu, mg_grid* out, mg_grid* pooled, const mg_bn_fused* bn);
bool bf16_bn_stats(mg_ctx*, const mg_grid* y, mg_sum* sums);
bool bf16_combine(mg_ctx*, const mg_grid* x, int relu_mask, const mg_grid* bn_x, int n_src, const mg_grad_src* src, mg_grid* d, mg_sum* sums);
bool bf16_bn_bwd_apply(mg_ctx*, const mg_grid* xraw, const mg_grid* d, mg_grid* out, const mg_sum* sums, int64_t count, const float* gamma,
                       const float* mean, const float* invstd, float* dgamma, float* dbeta, float* conv_dbias, float gscale);
int simt_dbias(mg_ctx* ctx, const mg_grid* g, int Cout, float* dbias, float gscale);
bool bf16_pool3(mg_ctx*, const mg_grid* in, mg_grid* out, uint8_t* code);
bool bf16_bn_relu_pool3(mg_ctx*, const mg_grid* z, const mg_bn_fused* bn, mg_grid* out, uint8_t* code);
bool bf16_import_nchw(mg_ctx*, const float* src, mg_grid* dst);
bool bf16_avgpool(mg_ctx*, const mg_grid* in, int r, mg_grid* out);
bool bf16_pool2(mg_ctx*, const mg_grid* in, mg_grid* out, int c_off);
bool bf16_dropout_forward(mg_ctx*, const DropK& k, int n_seg, const mg_grid* seg, const int32_t* mode, mg_grid* out);
bool bf16_dropout_backward(mg_ctx*, const DropK& k, mg_grid* g);

namespace {

constexpr int EB = 256;

// ---------------------------------------------------------------- import / export ---
template <typename T>
__global__ void import_nchw_kernel(const float* __restrict__ src, T* __restrict__ dst, int N, int C, int Cp, int H, int W) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)N * H * W * Cp;
  if (i >= total) return;
  int c = i % Cp; int64_t p = i / Cp;
  int x = p % W; p /= W; int y = p % H; int n = p / H;
  float v = c < C ? src[(((size_t)n * C + c) * H + y) * W + x] : 0.f;
  mg_st(dst + i, v);
}

template <typename T>
__global__ void export_nchw_kernel(GridV<T> g, float* __restrict__ dst) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)g.N * g.C * g.H * g.W;
  if (i >= total) return;
  int x = i % g.W; int64_t p = i / g.W;
  int y = p % g.H; p /= g.H; int c = p % g.C; int n = p / g.C;
  dst[i] = g.at(n, y, x, c);
}

// ---------------------------------------------------------------- BN finalise -------
__global__ void bn_finalize_kernel(const mg_sum* sums, int64_t count, int C, int Cp, const float* gamma,
                                   const float* beta, float* rmean, float* rvar, float eps, float momentum,
                                   int training, float* scale, float* shift, float* smean, float* sinvstd) {
  pdl_launch();
  pdl_wait();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cp) return;
  if (c >= C) { scale[c] = 0.f; shift[c] = 0.f; if (smean) { smean[c] = 0.f; sinvstd[c] = 0.f; } return; }
  double mean, var;
  if (training) {
    mean = mg_sum_get(sums[c]) / (double)count;
    var = mg_sum_get(sums[C + c]) / (double)count - mean * mean;   // biased
    if (var < 0) var = 0;
    if (rmean) {
      double unb = count > 1 ? var * (double)count / (double)(count - 1) : var;
      rmean[c] = (float)((1.0 - momentum) * rmean[c] + momentum * mean);
      rvar[c] = (float)((1.0 - momentum) * rvar[c] + momentum * unb);
    }
  } else {
    mean = rmean[c]; var = rvar[c];
  }
  double invstd = 1.0 / sqrt(var + (double)eps);
  float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
  scale[c] = (float)(g * invstd);
  shift[c] = (float)(b - g * invstd * mean);
  if (smean) { smean[c] = (float)mean; sinvstd[c] = (float)invstd; }
}

// ---------------------------------------------------------------- residual ----------
template <typename T>
__global__ void residual_kernel(GridV<T> z, GridV<T> s, int has_s, int relu, T* __restrict__ out, int out_cp) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)z.N * z.H * z.W * out_cp;
  if (i >= total) return;
  int c = i % out_cp; int64_t p = i / out_cp;
  float v = 0.f;
  if (c < z.C) {
    v = mg_ld(z.data + p * z.Cp + c);
    if (z.scale) v = mg_xform(v, z.scale[c], z.shift[c], z.relu);
    if (has_s && c < s.C) {
      float sv = mg_ld(s.data + p * s.Cp + c);
      if (s.scale) sv = mg_xform(sv, s.scale[c], s.shift[c], s.relu);
      v += sv;
    }
    if (relu) v = fmaxf(v, 0.f);
  }
  mg_st(out + i, v);
}

// same, one thread per (2x2 output block, channel): also writes maxpool2x2_ceil(out)
template <typename T>
__global__ void residual_pool_kernel(GridV<T> z, GridV<T> s, int has_s, int relu, T* __restrict__ out, int out_cp,
                                     T* __restrict__ pooled, int p_cp, int Hp, int Wp) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)z.N * Hp * Wp * out_cp;
  if (i >= total) return;
  int c = i % out_cp; int64_t q = i / out_cp;
  int px = q % Wp; q /= Wp; int py = q % Hp; int n = q / Hp;
  float best = -INFINITY;
  for (int dy = 0; dy < 2; ++dy)
    for (int dx = 0; dx < 2; ++dx) {
      int y = 2 * py + dy, x = 2 * px + dx;
      if (y >= z.H || x >= z.W) continue;
      int64_t p = ((int64_t)n * z.H + y) * z.W + x;
      float v = 0.f;
      if (c < z.C) {
        v = mg_ld(z.data + p * z.Cp + c);
        if (z.scale) v = mg_xform(v, z.scale[c], z.shift[c], z.relu);
        if (has_s && c < s.C) {
          float sv = mg_ld(s.data + p * s.Cp + c);
          if (s.scale) sv = mg_xform(sv, s.scale[c], s.shift[c], s.relu);
          v += sv;
        }
        if (relu) v = fmaxf(v, 0.f);
      }
      T r; mg_st(&r, v);
      out[p * out_cp + c] = r;
      float vr = mg_ld(&r);   // pool the stored (rounded) value: what a later gather would read
      if (vr > best || vr != vr) best = vr;
    }
  if (c < p_cp) mg_st(pooled + (((int64_t)n * Hp + py) * Wp + px) * p_cp + c, c < z.C ? best : 0.f);
}

// per-channel sum / sum of squares of a stored grid
template <typename T>
__global__ void __launch_bounds__(256) bn_stats_kernel(const T* __restrict__ y, int cp, int C, int64_t P, int pix_per_block,
                                                       mg_sum* sums) {
  const int cl = threadIdx.x % 32, lane = threadIdx.x / 32;
  const int c = blockIdx.y * 32 + cl;
  const int64_t p0 = (int64_t)blockIdx.x * pix_per_block, p1 = min(P, p0 + pix_per_block);
  float s = 0.f, s2 = 0.f;
  if (c < C)
    for (int64_t p = p0 + lane; p < p1; p += 8) { float v = mg_ld(y + p * cp + c); s += v; s2 = fmaf(v, v, s2); }
  __shared__ float red[2][8][33];
  red[0][lane][cl] = s; red[1][lane][cl] = s2;
  __syncthreads();
  if (lane == 0 && c < C) {
    float a = 0.f, b = 0.f;
    for (int l = 0; l < 8; ++l) { a += red[0][l][cl]; b += red[1][l][cl]; }
    mg_sum_add(sums + c, (double)a);
    mg_sum_add(sums + C + c, (double)b);
  }
}

// ---------------------------------------------------------------- pooling -----------
template <typename T>
__global__ void pool2_kernel(GridV<T> in, T* __restrict__ out, int Ho, int Wo, int out_cp, int c_off, int32_t* argmax) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)in.N * Ho * Wo * in.C;
  if (i >= total) return;
  int c = i % in.C; int64_t p = i / in.C;
  int px = p % Wo; int64_t q = p / Wo; int py = q % Ho; int n = q / Ho;
  int arg;
  float v = in.pooled(n, py, px, c, &arg);
  mg_st(out + p * out_cp + c_off + c, v);
  if (argmax) argmax[i] = arg;
}

template <typename T>
__global__ void copy_channels_kernel(GridV<T> in, T* __restrict__ out, int out_cp, int c_off) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)in.N * in.H * in.W * in.C;
  if (i >= total) return;
  int c = i % in.C; int64_t p = i / in.C;
  float v = mg_ld(in.data + p * in.Cp + c);
  if (in.scale) v = mg_xform(v, in.scale[c], in.shift[c], in.relu);
  mg_st(out + p * out_cp + c_off + c, v);
}

template <typename T>
__global__ void avgpool_kernel(GridV<T> in, int r, T* __restrict__ out, int Ho, int Wo, int out_cp) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)in.N * Ho * Wo * out_cp;
  if (i >= total) return;
  int c = i % out_cp; int64_t p = i / out_cp;
  int px = p % Wo; int64_t q = p / Wo; int py = q % Ho; int n = q / Ho;
  float s = 0.f;
  if (c < in.C) {
    for (int dy = 0; dy < r; ++dy)
      for (int dx = 0; dx < r; ++dx) s += in.at(n, py * r + dy, px * r + dx, c);
    s /= (float)(r * r);
  }
  mg_st(out + i, s);
}

// SpatialMaxPooling(3,3,2,2,1,1): floor mode, windows clipped to the image
template <typename T>
__device__ __forceinline__ float pool3_window(const GridV<T>& in, int n, int oy, int ox, int c, int* arg) {
  int y0 = max(oy * 2 - 1, 0), x0 = max(ox * 2 - 1, 0);
  int y1 = min(oy * 2 + 2, in.H), x1 = min(ox * 2 + 2, in.W);
  float best = -INFINITY; int bi = y0 * in.W + x0;
  for (int yy = y0; yy < y1; ++yy)
    for (int xx = x0; xx < x1; ++xx) {
      float v = in.at(n, yy, xx, c);
      if (v > best || v != v) { best = v; bi = yy * in.W + xx; }
    }
  *arg = bi;
  return best;
}

template <typename T>
__global__ void pool3_kernel(GridV<T> in, T* __restrict__ out, int Ho, int Wo, int out_cp) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)in.N * Ho * Wo * out_cp;
  if (i >= total) return;
  int c = i % out_cp; int64_t p = i / out_cp;
  int px = p % Wo; int64_t q = p / Wo; int py = q % Ho; int n = q / Ho;
  int arg; float v = 0.f;
  if (c < in.C) v = pool3_window(in, n, py, px, c, &arg);
  mg_st(out + i, v);
}

template <typename T>
__global__ void global_avgpool_kernel(GridV<T> in, T* __restrict__ out, int out_cp) {
  int i = blockIdx.x * EB + threadIdx.x;
  if (i >= in.N * out_cp) return;
  int c = i % out_cp, n = i / out_cp;
  float s = 0.f;
  if (c < in.C) {
    for (int y = 0; y < in.H; ++y)
      for (int x = 0; x < in.W; ++x) s += in.at(n, y, x, c);
    s /= (float)(in.H * in.W);
  }
  mg_st(out + i, s);
}

template <typename T>
__global__ void global_avgpool_bwd_kernel(const T* __restrict__ dout, int dout_cp, T* __restrict__ din, int N, int H, int W, int C, int Cp) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)N * H * W * Cp;
  if (i >= total) return;
  int c = i % Cp; int64_t p = i / Cp; int n = p / (H * W);
  float v = c < C ? mg_ld(dout + (size_t)n * dout_cp + c) / (float)(H * W) : 0.f;
  mg_st(din + i, v);
}

// ---------------------------------------------------------------- gradient combine --
template <typename T>
struct SrcV { GridV<T> g; int c_off; int mode; };

template <typename T>
struct CombineP {
  GridV<T> x;
  int relu_mask;
  const T* bn_x; int bn_cp;
  int n_src; SrcV<T> src[MG_MAX_SRC];
  T* d; int d_cp;
  mg_sum* bn_sums;
  int pix_per_block;
};

// block = 32 channels x 8 pixel lanes
template <typename T>
__global__ void __launch_bounds__(256) combine_kernel(CombineP<T> p) {
  const int cl = threadIdx.x % 32, lane = threadIdx.x / 32;
  const int c = blockIdx.y * 32 + cl;
  const int64_t P = (int64_t)p.x.N * p.x.H * p.x.W;
  const int64_t p0 = (int64_t)blockIdx.x * p.pix_per_block;
  const int64_t p1 = min(P, p0 + p.pix_per_block);
  const GridV<T>& X = p.x;
  float sd = 0.f, sdx = 0.f;
  if (c < p.d_cp) {
    for (int64_t pix = p0 + lane; pix < p1; pix += 8) {
      float sum = 0.f;
      if (c < X.C) {
        int x = pix % X.W; int64_t q = pix / X.W; int y = q % X.H; int n = q / X.H;
        for (int s = 0; s < p.n_src; ++s) {
          const GridV<T>& G = p.src[s].g;
          const int gc = p.src[s].c_off + c;
          const int mode = p.src[s].mode;
          if (mode == MG_SEG_SAME) {
            sum += G.raw(n, y, x, gc);
          } else if (mode == MG_SEG_UP) {
            sum += G.raw(n, 2 * y, 2 * x, gc) + G.raw(n, 2 * y, 2 * x + 1, gc) +
                   G.raw(n, 2 * y + 1, 2 * x, gc) + G.raw(n, 2 * y + 1, 2 * x + 1, gc);
          } else if (mode == MG_SEG_POOL) {
            int arg; X.pooled(n, y >> 1, x >> 1, c, &arg);
            if (arg == y * X.W + x) sum += G.raw(n, y >> 1, x >> 1, gc);
          } else {  // 3x3 stride-2 pad-1 windows containing (y, x)
            int oy0 = max((y - 1 + 1) / 2, 0), oy1 = min((y + 1) / 2, G.H - 1);
            int ox0 = max((x - 1 + 1) / 2, 0), ox1 = min((x + 1) / 2, G.W - 1);
            for (int oy = oy0; oy <= oy1; ++oy)
              for (int ox = ox0; ox <= ox1; ++ox) {
                int arg; pool3_window(X, n, oy, ox, c, &arg);
                if (arg == y * X.W + x) sum += G.raw(n, oy, ox, gc);
              }
          }
        }
        if (p.relu_mask) { float v = X.at(n, y, x, c); if (!(v > 0.f)) sum = 0.f; }
        if (p.bn_sums) { sd += sum; sdx += sum * mg_ld(p.bn_x + pix * p.bn_cp + c); }
      }
      mg_st(p.d + pix * p.d_cp + c, sum);
    }
  }
  if (p.bn_sums) {
    __shared__ float red[2][8][33];
    red[0][lane][cl] = sd; red[1][lane][cl] = sdx;
    __syncthreads();
    if (lane == 0 && c < X.C) {
      float a = 0.f, b = 0.f;
      for (int l = 0; l < 8; ++l) { a += red[0][l][cl]; b += red[1][l][cl]; }
      mg_sum_add(p.bn_sums + c, (double)a);
      mg_sum_add(p.bn_sums + X.C + c, (double)b);
    }
  }
}

// ---------------------------------------------------------------- BN backward -------
// coef[0*Cp+c]=A, [1*Cp+c]=B, [2*Cp+c]=Cc with d' = A*d + B*xraw + Cc
__global__ void bn_bwd_coef_kernel(const mg_sum* sums, int64_t count, int C, int Cp, const float* gamma,
                                   const float* mean, const float* invstd, float* dgamma, float* dbeta,
                                   float gscale, float* coef, float* conv_dbias) {
  pdl_launch();
  pdl_wait();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cp) return;
  if (c >= C) { coef[c] = 0.f; coef[Cp + c] = 0.f; coef[2 * Cp + c] = 0.f; return; }
  double sd = mg_sum_get(sums[c]), sdx = mg_sum_get(sums[C + c]);
  double mu = mean[c], is = invstd[c], g = gamma ? gamma[c] : 1.0;
  double dg = is * (sdx - mu * sd);
  if (dgamma) dgamma[c] += gscale * (float)dg;
  if (dbeta) dbeta[c] += gscale * (float)sd;
  double n = (double)count;
  const double Ad = g * is, Bd = -g * is * is * dg / n, Cd = g * is * (mu * is * dg / n - sd / n);
  coef[c] = (float)Ad;
  coef[Cp + c] = (float)Bd;
  coef[2 * Cp + c] = (float)Cd;
  // gradBias of the convolution that produced xraw = sum over pixels of the result = A*sum d + B*sum xraw + C*n
  // (identically zero in exact arithmetic: pure rounding noise in the reference as well)
  if (conv_dbias) conv_dbias[c] += gscale * (float)(Ad * sd + Bd * (mu * n) + Cd * n);
}

template <typename T>
__global__ void bn_bwd_apply_kernel(const T* __restrict__ xraw, int x_cp, const T* d, int d_cp, T* out, int o_cp, int C,
                                    int64_t P, const float* __restrict__ coef) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  if (i >= P * o_cp) return;
  int c = i % o_cp; int64_t pix = i / o_cp;
  float v = 0.f;
  if (c < C)
    v = fmaf(coef[c], mg_ld(d + pix * d_cp + c), fmaf(coef[d_cp + c], mg_ld(xraw + pix * x_cp + c), coef[2 * d_cp + c]));
  mg_st(out + i, v);
}

// ---------------------------------------------------------------- input path: crop / flip / normalise ----------
// dst[n][c][y][x] = (src[n][c][y0[n] + y][x0[n] + (flip[n] ? oW-1-x : x)] - mean[c]) / std[c], zero where the window leaves
// the source image (the reference's test hook pads its centre crop with zeros, dataset/cifar100-whitened/donkey.lua:172-174)
__global__ void crop_flip_normalize_kernel(const float* __restrict__ src, int C, int H, int W, float* __restrict__ dst, int oH, int oW,
                                           const int32_t* __restrict__ y0, const int32_t* __restrict__ x0, const int32_t* __restrict__ flip,
                                           const float* __restrict__ mean, const float* __restrict__ stdv, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  if (i >= total) return;
  const int x = (int)(i % oW); int64_t q = i / oW;
  const int y = (int)(q % oH); q /= oH;
  const int c = (int)(q % C); const int n = (int)(q / C);
  const int sx = (x0 ? x0[n] : 0) + ((flip && flip[n]) ? oW - 1 - x : x), sy = (y0 ? y0[n] : 0) + y;
  float v = 0.f;
  if (sx >= 0 && sx < W && sy >= 0 && sy < H) {
    v = src[(((int64_t)n * C + c) * H + sy) * W + sx];
    if (mean) v -= mean[c];
    if (stdv) v /= stdv[c];
  }
  dst[i] = v;
}

// ---------------------------------------------------------------- criteria ----------
// The scalar loss is accumulated as a deterministic integer sum (mg_sum scratch of the context, left zeroed) and added to the
// caller's float by loss_finalize_kernel: the reported loss is bit-identical from run to run.
__global__ void loss_finalize_kernel(mg_sum* acc, float* loss) {
  *loss += (float)mg_sum_get(*acc);
  acc->hi = 0; acc->lo = 0;
}

// one block per sample: LogSoftMax + ClassNLLCriterion(mean) forward and gradient
template <typename T>
__global__ void nll_kernel(const T* __restrict__ logits, int C, int ld, const int32_t* __restrict__ target,
                           float* logprob, mg_sum* loss, T* dlogits, int dl_ld, float gscale, int N) {
  int n = blockIdx.x;
  const T* row = logits + (size_t)n * ld;
  __shared__ float red[32];
  float m = -INFINITY;
  for (int c = threadIdx.x; c < C; c += blockDim.x) m = fmaxf(m, mg_ld(row + c));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = m;
  __syncthreads();
  m = red[0];
  for (int w = 1; w < blockDim.x / 32; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s += expf(mg_ld(row + c) - m);
  s = warp_sum(s);
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = s;
  __syncthreads();
  s = 0.f;
  for (int w = 0; w < blockDim.x / 32; ++w) s += red[w];
  float lse = m + logf(s);
  int t = target[n];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float lp = mg_ld(row + c) - lse;
    if (logprob) logprob[(size_t)n * C + c] = lp;
    if (dlogits) mg_st(dlogits + (size_t)n * dl_ld + c, gscale * (expf(lp) - (c == t ? 1.f : 0.f)) / (float)N);
  }
  if (threadIdx.x == 0 && loss) mg_sum_add(loss, (double)(-(mg_ld(row + t) - lse) / (float)N));
}

// Sigmoid + BCECriterion (mean over all elements, eps 1e-12)
template <typename T>
__global__ void bce_kernel(GridV<T> x, const float* __restrict__ target, float* prob, mg_sum* loss, T* dx, int dx_cp, float gscale) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)x.N * x.C * x.H * x.W;
  float l = 0.f;
  if (i < total) {
    int xx = i % x.W; int64_t p = i / x.W;
    int y = p % x.H; p /= x.H; int c = p % x.C; int n = p / x.C;
    float v = x.at(n, y, xx, c);
    float pr = 1.f / (1.f + expf(-v));
    float t = target[i];
    const float eps = 1e-12f;
    l = -(logf(pr + eps) * t + logf(1.f - pr + eps) * (1.f - t)) / (float)total;
    if (prob) prob[i] = pr;
    if (dx) {
      float dp = -(t - pr) / ((1.f - pr + eps) * (pr + eps)) / (float)total;
      mg_st(dx + (((size_t)n * x.H + y) * x.W + xx) * dx_cp + c, gscale * dp * pr * (1.f - pr));
    }
  }
  l = warp_sum(l);
  if (loss && threadIdx.x % 32 == 0 && l != 0.f) mg_sum_add(loss, (double)l);
}

__global__ void sgd_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ v, int64_t n,
                           float lr, float mu, float wd, int first) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  if (i >= n) return;
  float gi = fmaf(wd, w[i], g[i]);
  float vi = first ? gi : fmaf(mu, v[i], gi);
  v[i] = vi;
  w[i] = fmaf(-lr, vi, w[i]);
}

// ---------------------------------------------------------------- dropout -----------
// one thread per (pixel, 4 channels of the pitch); the logical elements of a quad span at most two Philox calls
template <typename T>
__global__ void dropout_fwd_kernel(DropSegs<T> d, DropK k, T* __restrict__ out, int N, int H, int W, int C, int Cp) {
  const int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  const int Q = Cp / 4;
  if (i >= (int64_t)N * H * W * Q) return;
  const int q = i % Q; const int64_t pix = i / Q;
  const int x = pix % W; const int64_t r = pix / W; const int y = r % H; const int n = r / H;
  const int c0 = q * 4, nl = min(4, C - c0);   // logical channels of the quad (none: pad only)
  const uint32_t keep = nl > 0 ? drop_keep_bits((uint64_t)pix * C + c0, nl, k) : 0u;
  for (int e = 0; e < 4; ++e) {
    float v = 0.f;
    if (e < nl && (keep >> e & 1u)) v = drop_gather(d, n, y, x, c0 + e) * k.s;
    mg_st(out + pix * Cp + c0 + e, v);
  }
}

template <typename T>
__global__ void dropout_bwd_kernel(DropK k, T* __restrict__ g, int64_t P, int C, int Cp) {
  const int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  const int Q = Cp / 4;
  if (i >= P * Q) return;
  const int q = i % Q; const int64_t pix = i / Q;
  const int c0 = q * 4, nl = min(4, C - c0);
  if (nl <= 0) return;
  const uint32_t keep = drop_keep_bits((uint64_t)pix * C + c0, nl, k);
  for (int e = 0; e < nl; ++e) {
    T* p = g + pix * Cp + c0 + e;
    mg_st(p, (keep >> e & 1u) ? mg_ld(p) * k.s : 0.f);
  }
}

__global__ void dropout_advance_kernel(uint64_t* step) { ++*step; }

}  // namespace

// mask parameters of a dropout call; rejects p outside [0, 1)
static int drop_key(mg_ctx* ctx, const mg_dropout* dp, DropK* k) {
  MG_REQUIRE(ctx, dp->p >= 0.f && dp->p < 1.f, MG_ERR_INVALID_ARG, "dropout: p = %g is outside [0, 1)", (double)dp->p);
  MG_REQUIRE(ctx, dp->step != nullptr, MG_ERR_INVALID_ARG, "dropout: null step counter");
  k->key_lo = (uint32_t)dp->seed; k->key_hi = (uint32_t)(dp->seed >> 32);
  k->op = dp->op; k->rank = dp->rank; k->step = dp->step;
  k->t = (uint32_t)std::min(floor((double)dp->p * 4294967296.0), 4294967295.0);
  k->s = (float)(1.0 / (1.0 - (double)dp->p));
  return MG_OK;
}

#define GRID1(total) (unsigned)mg_cdiv((int64_t)(total), EB)

extern "C" {

int mg_import_nchw(mg_ctx* ctx, const float* src, mg_grid* dst) {
  if (!ctx || !src || !dst) return MG_ERR_INVALID_ARG;
  if (ctx->dtype == MG_BF16 && bf16_import_nchw(ctx, src, dst)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  int64_t total = (int64_t)dst->N * dst->H * dst->W * dst->Cp;
  MG_DISPATCH(ctx, import_nchw_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(src, (T*)dst->data, dst->N, dst->C, dst->Cp, dst->H, dst->W););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_export_nchw(mg_ctx* ctx, const mg_grid* src, float* dst) {
  if (!ctx || !src || !dst) return MG_ERR_INVALID_ARG;
  int64_t total = (int64_t)src->N * src->H * src->W * src->C;
  MG_DISPATCH(ctx, export_nchw_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*src), dst););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_bn_finalize(mg_ctx* ctx, const mg_sum* bn_sums, int64_t count, int32_t C, int32_t Cp, const float* gamma,
                   const float* beta, float* running_mean, float* running_var, float eps, float momentum,
                   int training, float* scale, float* shift, float* save_mean, float* save_invstd) {
  if (!ctx || !scale || !shift) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, training ? bn_sums != nullptr : (running_mean && running_var), MG_ERR_INVALID_ARG,
             "bn_finalize: missing statistics");
  mg_launch_pdl(bn_finalize_kernel, dim3((unsigned)mg_cdiv(Cp, 128)), dim3(128), 0, ctx->stream, bn_sums, count, (int)C, (int)Cp, gamma, beta,
                running_mean, running_var, eps, momentum, training, scale, shift, save_mean, save_invstd);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_residual_forward(mg_ctx* ctx, const mg_grid* z, const mg_grid* s, int relu, mg_grid* out, mg_grid* pooled) {
  if (!ctx || !z || !out) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, out->N == z->N && out->H == z->H && out->W == z->W && out->C == z->C, MG_ERR_SHAPE, "residual: out shape");
  if (s) MG_REQUIRE(ctx, s->N == z->N && s->H == z->H && s->W == z->W && s->C <= z->C, MG_ERR_SHAPE,
                    "residual: shortcut %dx%dx%d vs %dx%dx%d", s->H, s->W, s->C, z->H, z->W, z->C);
  if (pooled) {
    int Hp = (z->H + 1) / 2, Wp = (z->W + 1) / 2;
    MG_REQUIRE(ctx, pooled->N == z->N && pooled->H == Hp && pooled->W == Wp && pooled->C == z->C && pooled->Cp <= out->Cp,
               MG_ERR_SHAPE, "residual: pooled shape");
  }
  if (ctx->dtype == MG_BF16 && bf16_apply(ctx, z, s, relu, out, pooled, nullptr)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  if (pooled) {
    int Hp = (z->H + 1) / 2, Wp = (z->W + 1) / 2;
    int64_t total = (int64_t)z->N * Hp * Wp * out->Cp;
    MG_DISPATCH(ctx, residual_pool_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*z), s ? make_view<T>(*s) : make_view<T>(*z),
                                                                                  s != nullptr, relu, (T*)out->data, out->Cp,
                                                                                  (T*)pooled->data, pooled->Cp, Hp, Wp););
    MG_CHECK_LAUNCH(ctx);
    return MG_OK;
  }
  int64_t total = (int64_t)z->N * z->H * z->W * out->Cp;
  MG_DISPATCH(ctx, residual_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*z), s ? make_view<T>(*s) : make_view<T>(*z),
                                                                           s != nullptr, relu, (T*)out->data, out->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_bn_residual_forward(mg_ctx* ctx, const mg_grid* z, const mg_bn_fused* bn, const mg_grid* s, int relu, mg_grid* out, mg_grid* pooled) {
  if (!ctx || !z || !bn || !out) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, z->scale && z->shift, MG_ERR_INVALID_ARG, "bn_residual: z needs scale / shift workspaces");
  MG_REQUIRE(ctx, bn->training ? bn->sums != nullptr : (bn->running_mean && bn->running_var), MG_ERR_INVALID_ARG,
             "bn_residual: missing statistics");
  MG_REQUIRE(ctx, out->N == z->N && out->H == z->H && out->W == z->W && out->C == z->C, MG_ERR_SHAPE, "bn_residual: out shape");
  if (s) MG_REQUIRE(ctx, s->N == z->N && s->H == z->H && s->W == z->W && s->C <= z->C, MG_ERR_SHAPE,
                    "bn_residual: shortcut %dx%dx%d vs %dx%dx%d", s->H, s->W, s->C, z->H, z->W, z->C);
  if (pooled)
    MG_REQUIRE(ctx, pooled->N == z->N && pooled->H == (z->H + 1) / 2 && pooled->W == (z->W + 1) / 2 && pooled->C == z->C && pooled->Cp <= out->Cp,
               MG_ERR_SHAPE, "bn_residual: pooled shape");
  if (ctx->dtype == MG_BF16 && bf16_apply(ctx, z, s, relu, out, pooled, bn)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  int rc = mg_bn_finalize(ctx, bn->sums, bn->count, z->C, z->Cp, bn->gamma, bn->beta, bn->running_mean, bn->running_var, bn->eps,
                          bn->momentum, bn->training, const_cast<float*>(z->scale), const_cast<float*>(z->shift), bn->save_mean, bn->save_invstd);
  if (rc) return rc;
  return mg_residual_forward(ctx, z, s, relu, out, pooled);
}

int mg_bn_relu_pool3_forward(mg_ctx* ctx, const mg_grid* z, const mg_bn_fused* bn, mg_grid* out, uint8_t* argmax_code) {
  if (!ctx || !z || !bn || !out || !argmax_code) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, z->scale && z->shift, MG_ERR_INVALID_ARG, "bn_relu_pool3: z needs scale / shift workspaces");
  MG_REQUIRE(ctx, bn->training ? bn->sums != nullptr : (bn->running_mean && bn->running_var), MG_ERR_INVALID_ARG, "bn_relu_pool3: missing statistics");
  MG_REQUIRE(ctx, out->N == z->N && out->H == (z->H - 1) / 2 + 1 && out->W == (z->W - 1) / 2 + 1 && out->C == z->C, MG_ERR_SHAPE,
             "bn_relu_pool3: out %dx%dx%d for %dx%dx%d", out->H, out->W, out->C, z->H, z->W, z->C);
  MG_REQUIRE(ctx, ctx->dtype == MG_BF16, MG_ERR_UNSUPPORTED, "bn_relu_pool3: bf16 contexts only (fp32 runs mg_bn_residual_forward + mg_pool3s2_forward)");
  MG_REQUIRE(ctx, bf16_bn_relu_pool3(ctx, z, bn, out, argmax_code), MG_ERR_UNSUPPORTED, "bn_relu_pool3: unsupported layout");
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_bn_stats(mg_ctx* ctx, const mg_grid* y, mg_sum* bn_sums) {
  if (!ctx || !y || !bn_sums) return MG_ERR_INVALID_ARG;
  if (ctx->dtype == MG_BF16 && bf16_bn_stats(ctx, y, bn_sums)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  int64_t P = (int64_t)y->N * y->H * y->W;
  int ppb = (int)std::max<int64_t>(64, mg_cdiv(P, (int64_t)ctx->num_sms * 8));
  dim3 grid((unsigned)mg_cdiv(P, ppb), (unsigned)mg_cdiv(y->C, 32));
  MG_DISPATCH(ctx, bn_stats_kernel<T><<<grid, 256, 0, ctx->stream>>>((const T*)y->data, y->Cp, y->C, P, ppb, bn_sums););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_memset_zero(mg_ctx* ctx, void* ptr, size_t bytes) {
  if (!ctx || !ptr) return MG_ERR_INVALID_ARG;
  MG_CUDA(ctx, cudaMemsetAsync(ptr, 0, bytes, ctx->stream));
  return MG_OK;
}

int mg_pool_forward(mg_ctx* ctx, const mg_grid* in, mg_grid* out, int32_t c_offset, int32_t* argmax) {
  if (!ctx || !in || !out) return MG_ERR_INVALID_ARG;
  int Ho = (in->H + 1) / 2, Wo = (in->W + 1) / 2;
  MG_REQUIRE(ctx, out->H == Ho && out->W == Wo && out->N == in->N && c_offset + in->C <= out->Cp, MG_ERR_SHAPE,
             "pool: out %dx%d (C %d) for in %dx%d (C %d, off %d)", out->H, out->W, out->C, in->H, in->W, in->C, c_offset);
  if (ctx->dtype == MG_BF16 && !argmax && bf16_pool2(ctx, in, out, c_offset)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  int64_t total = (int64_t)in->N * Ho * Wo * in->C;
  MG_DISPATCH(ctx, pool2_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*in), (T*)out->data, Ho, Wo, out->Cp, c_offset, argmax););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_copy_channels(mg_ctx* ctx, const mg_grid* in, mg_grid* out, int32_t c_offset) {
  if (!ctx || !in || !out) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, out->H == in->H && out->W == in->W && out->N == in->N && c_offset + in->C <= out->Cp, MG_ERR_SHAPE, "copy_channels: shape");
  int64_t total = (int64_t)in->N * in->H * in->W * in->C;
  MG_DISPATCH(ctx, copy_channels_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*in), (T*)out->data, out->Cp, c_offset););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_dropout_forward(mg_ctx* ctx, const mg_dropout* dp, int32_t n_seg, const mg_grid* seg, const int32_t* seg_mode, mg_grid* out) {
  if (!ctx || !dp || !seg || !seg_mode || !out || !out->data || n_seg < 1 || n_seg > MG_MAX_SEG) return MG_ERR_INVALID_ARG;
  DropK k;
  int rc = drop_key(ctx, dp, &k);
  if (rc) return rc;
  int C = 0;
  for (int s = 0; s < n_seg; ++s) {
    const mg_grid& g = seg[s];
    MG_REQUIRE(ctx, seg_mode[s] == MG_SEG_SAME || seg_mode[s] == MG_SEG_UP, MG_ERR_INVALID_ARG, "dropout_forward: segment %d mode %d", s, seg_mode[s]);
    const int f = seg_mode[s] == MG_SEG_UP ? 2 : 1;
    MG_REQUIRE(ctx, g.data && g.N == out->N && f * g.H == out->H && f * g.W == out->W && g.C <= g.Cp, MG_ERR_SHAPE,
               "dropout_forward: segment %d (mode %d) is %dx%d, output %dx%d", s, seg_mode[s], g.H, g.W, out->H, out->W);
    C += g.C;
  }
  MG_REQUIRE(ctx, C == out->C && out->Cp >= out->C && out->Cp % 8 == 0, MG_ERR_SHAPE, "dropout_forward: %d channels into C %d Cp %d", C, out->C, out->Cp);
  const int64_t P = (int64_t)out->N * out->H * out->W;
  MG_REQUIRE(ctx, P * C < ((int64_t)1 << 34), MG_ERR_SHAPE, "dropout_forward: %lld elements exceed the 2^34 of the Philox counter", (long long)(P * C));
  if (ctx->dtype == MG_BF16 && bf16_dropout_forward(ctx, k, n_seg, seg, seg_mode, out)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  MG_DISPATCH(ctx, dropout_fwd_kernel<T><<<GRID1(P * (out->Cp / 4)), EB, 0, ctx->stream>>>(make_drop_segs<T>(n_seg, seg, seg_mode), k, (T*)out->data,
                                                                                        out->N, out->H, out->W, out->C, out->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_dropout_backward(mg_ctx* ctx, const mg_dropout* dp, mg_grid* g) {
  if (!ctx || !dp || !g || !g->data) return MG_ERR_INVALID_ARG;
  DropK k;
  int rc = drop_key(ctx, dp, &k);
  if (rc) return rc;
  MG_REQUIRE(ctx, g->Cp >= g->C && g->Cp % 8 == 0, MG_ERR_SHAPE, "dropout_backward: C %d Cp %d", g->C, g->Cp);
  const int64_t P = (int64_t)g->N * g->H * g->W;
  MG_REQUIRE(ctx, P * g->C < ((int64_t)1 << 34), MG_ERR_SHAPE, "dropout_backward: %lld elements exceed the 2^34 of the Philox counter", (long long)(P * g->C));
  if (ctx->dtype == MG_BF16 && bf16_dropout_backward(ctx, k, g)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  MG_DISPATCH(ctx, dropout_bwd_kernel<T><<<GRID1(P * (g->Cp / 4)), EB, 0, ctx->stream>>>(k, (T*)g->data, P, g->C, g->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_dropout_advance(mg_ctx* ctx, uint64_t* step) {
  if (!ctx || !step) return MG_ERR_INVALID_ARG;
  dropout_advance_kernel<<<1, 1, 0, ctx->stream>>>(step);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_im2col(mg_ctx* ctx, const mg_grid* in, int32_t ksize, int32_t stride, int32_t pad, mg_grid* col) {
  if (!ctx || !in || !col || !in->data || !col->data || ksize < 1 || stride < 1 || pad < 0) return MG_ERR_INVALID_ARG;
  const int Ho = (in->H + 2 * pad - ksize) / stride + 1, Wo = (in->W + 2 * pad - ksize) / stride + 1;
  MG_REQUIRE(ctx, col->N == in->N && col->H == Ho && col->W == Wo && col->C == in->C * ksize * ksize, MG_ERR_SHAPE,
             "im2col: col is %dx%dx%d, expected %dx%dx%d", col->H, col->W, col->C, Ho, Wo, in->C * ksize * ksize);
  MG_REQUIRE(ctx, ctx->dtype == MG_BF16, MG_ERR_UNSUPPORTED, "im2col: bf16 contexts only (the fp32 path convolves the image directly)");
  MG_REQUIRE(ctx, bf16_im2col(ctx, in, ksize, stride, pad, col), MG_ERR_UNSUPPORTED, "im2col: pending affine or unaligned channel pitch");
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_avgpool_forward(mg_ctx* ctx, const mg_grid* in, int32_t r, mg_grid* out) {
  if (!ctx || !in || !out || r < 1) return MG_ERR_INVALID_ARG;
  int Ho = in->H / r, Wo = in->W / r;
  MG_REQUIRE(ctx, out->H == Ho && out->W == Wo && out->N == in->N && out->C == in->C, MG_ERR_SHAPE, "avgpool: shape");
  if (ctx->dtype == MG_BF16 && bf16_avgpool(ctx, in, r, out)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  int64_t total = (int64_t)in->N * Ho * Wo * out->Cp;
  MG_DISPATCH(ctx, avgpool_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*in), r, (T*)out->data, Ho, Wo, out->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_pool3s2_forward(mg_ctx* ctx, const mg_grid* in, mg_grid* out, uint8_t* argmax_code) {
  if (!ctx || !in || !out) return MG_ERR_INVALID_ARG;
  int Ho = (in->H + 2 - 3) / 2 + 1, Wo = (in->W + 2 - 3) / 2 + 1;
  MG_REQUIRE(ctx, out->H == Ho && out->W == Wo && out->N == in->N && out->C == in->C, MG_ERR_SHAPE, "pool3s2: shape");
  if (ctx->dtype == MG_BF16 && bf16_pool3(ctx, in, out, argmax_code)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  MG_REQUIRE(ctx, argmax_code == nullptr, MG_ERR_UNSUPPORTED, "pool3s2: arg-max codes are only produced by the bf16 path");
  int64_t total = (int64_t)in->N * Ho * Wo * out->Cp;
  MG_DISPATCH(ctx, pool3_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*in), (T*)out->data, Ho, Wo, out->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_global_avgpool_forward(mg_ctx* ctx, const mg_grid* in, mg_grid* out) {
  if (!ctx || !in || !out) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, out->N == in->N && out->H == 1 && out->W == 1 && out->C == in->C, MG_ERR_SHAPE, "global_avgpool: shape");
  MG_DISPATCH(ctx, global_avgpool_kernel<T><<<GRID1(in->N * out->Cp), EB, 0, ctx->stream>>>(make_view<T>(*in), (T*)out->data, out->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_global_avgpool_backward(mg_ctx* ctx, const mg_grid* dout, mg_grid* din) {
  if (!ctx || !dout || !din) return MG_ERR_INVALID_ARG;
  int64_t total = (int64_t)din->N * din->H * din->W * din->Cp;
  MG_DISPATCH(ctx, global_avgpool_bwd_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>((const T*)dout->data, dout->Cp, (T*)din->data,
                                                                                     din->N, din->H, din->W, din->C, din->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_grad_combine(mg_ctx* ctx, const mg_grid* x, int relu_mask, const mg_grid* bn_x, int32_t n_src,
                    const mg_grad_src* src, mg_grid* d, mg_sum* bn_sums) {
  if (!ctx || !x || !d || n_src < 0 || n_src > MG_MAX_SRC || (n_src && !src)) return MG_ERR_INVALID_ARG;
  if (relu_mask == 2) {
    // the tensor itself was never stored (mg_bn_relu_pool3_forward): x is its 3x3 / stride-2 max-pooled form, the one source routes
    // through the arg-max codes, and the ReLU mask of an element is the sign of the pooled value it was the arg-max of
    MG_REQUIRE(ctx, n_src == 1 && src[0].mode == 3 && src[0].aux && bn_x, MG_ERR_INVALID_ARG, "combine: relu_mask 2 needs one arg-max-coded source and bn_x");
    MG_REQUIRE(ctx, x->N == d->N && x->C == d->C && x->H == (d->H - 1) / 2 + 1 && x->W == (d->W - 1) / 2 + 1 && src[0].g.H == x->H && src[0].g.W == x->W
               && bn_x->H == d->H && bn_x->W == d->W, MG_ERR_SHAPE, "combine: relu_mask 2 shapes");
    MG_REQUIRE(ctx, ctx->dtype == MG_BF16 && bf16_combine(ctx, x, relu_mask, bn_x, n_src, src, d, bn_sums), MG_ERR_UNSUPPORTED, "combine: relu_mask 2 is a bf16 fast path");
    MG_CHECK_LAUNCH(ctx);
    return MG_OK;
  }
  MG_REQUIRE(ctx, d->N == x->N && d->H == x->H && d->W == x->W && d->C == x->C, MG_ERR_SHAPE, "combine: d shape");
  for (int s = 0; s < n_src; ++s) {
    const mg_grid& g = src[s].g;
    int m = src[s].mode;
    bool ok = g.N == x->N && src[s].c_offset + x->C <= g.Cp;
    if (m == MG_SEG_SAME) ok = ok && g.H == x->H && g.W == x->W;
    else if (m == MG_SEG_UP) ok = ok && g.H == 2 * x->H && g.W == 2 * x->W;
    else if (m == MG_SEG_POOL) ok = ok && g.H == (x->H + 1) / 2 && g.W == (x->W + 1) / 2;
    else if (m == 3) ok = ok && g.H == (x->H - 1) / 2 + 1 && g.W == (x->W - 1) / 2 + 1;
    else ok = false;
    MG_REQUIRE(ctx, ok, MG_ERR_SHAPE, "combine: src %d (mode %d, %dx%dx%d off %d) does not match x %dx%dx%d", s, m, g.H,
               g.W, g.Cp, src[s].c_offset, x->H, x->W, x->C);
  }
  if (ctx->dtype == MG_BF16 && bf16_combine(ctx, x, relu_mask, bn_x, n_src, src, d, bn_sums)) { MG_CHECK_LAUNCH(ctx); return MG_OK; }
  int64_t P = (int64_t)x->N * x->H * x->W;
  MG_DISPATCH(ctx, {
    CombineP<T> p;
    p.x = make_view<T>(*x); p.relu_mask = relu_mask;
    p.bn_x = (const T*)(bn_x ? bn_x->data : x->data); p.bn_cp = bn_x ? bn_x->Cp : x->Cp;
    p.n_src = n_src;
    for (int s = 0; s < n_src; ++s) { p.src[s].g = make_view<T>(src[s].g); p.src[s].c_off = src[s].c_offset; p.src[s].mode = src[s].mode; }
    p.d = (T*)d->data; p.d_cp = d->Cp; p.bn_sums = bn_sums;
    p.pix_per_block = 64;
    dim3 grid((unsigned)mg_cdiv(P, p.pix_per_block), (unsigned)mg_cdiv(d->Cp, 32));
    combine_kernel<T><<<grid, 256, 0, ctx->stream>>>(p);
  });
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_bn_backward(mg_ctx* ctx, const mg_grid* xraw, const mg_grid* d, mg_grid* out, const mg_sum* bn_sums, int64_t count,
                   const float* gamma, const float* save_mean, const float* save_invstd, float* dgamma, float* dbeta,
                   float gscale, float* coef_ws, float* conv_dbias) {
  if (!ctx || !xraw || !d || !out || !bn_sums || !save_mean || !save_invstd || !coef_ws) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, d->N == xraw->N && d->H == xraw->H && d->W == xraw->W && d->C == xraw->C, MG_ERR_SHAPE, "bn_backward: shape");
  MG_REQUIRE(ctx, out->N == d->N && out->H == d->H && out->W == d->W && out->C == d->C, MG_ERR_SHAPE, "bn_backward: out shape");
  // bf16: one pass (coefficients derived in-kernel, block 0 accumulates dgamma / dbeta)
  if (ctx->dtype == MG_BF16 && bf16_bn_bwd_apply(ctx, xraw, d, out, bn_sums, count, gamma, save_mean, save_invstd, dgamma, dbeta, conv_dbias, gscale)) {
    MG_CHECK_LAUNCH(ctx);
    return MG_OK;
  }
  mg_launch_pdl(bn_bwd_coef_kernel, dim3((unsigned)mg_cdiv(d->Cp, 128)), dim3(128), 0, ctx->stream, bn_sums, count, (int)d->C, (int)d->Cp, gamma,
                save_mean, save_invstd, dgamma, dbeta, gscale, coef_ws, conv_dbias);
  MG_CHECK_LAUNCH(ctx);
  int64_t P = (int64_t)d->N * d->H * d->W;
  MG_DISPATCH(ctx, bn_bwd_apply_kernel<T><<<GRID1(P * out->Cp), EB, 0, ctx->stream>>>((const T*)xraw->data, xraw->Cp, (const T*)d->data, d->Cp,
                                                                                      (T*)out->data, out->Cp, d->C, P, coef_ws););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_crop_flip_normalize(mg_ctx* ctx, const float* src, int32_t N, int32_t C, int32_t H, int32_t W, float* dst, int32_t oH, int32_t oW,
                           const int32_t* y0, const int32_t* x0, const int32_t* flip, const float* mean, const float* stdv) {
  if (!ctx || !src || !dst || N < 1 || C < 1 || H < 1 || W < 1 || oH < 1 || oW < 1) return MG_ERR_INVALID_ARG;
  const int64_t total = (int64_t)N * C * oH * oW;
  crop_flip_normalize_kernel<<<GRID1(total), EB, 0, ctx->stream>>>(src, C, H, W, dst, oH, oW, y0, x0, flip, mean, stdv, total);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_nll_forward_backward(mg_ctx* ctx, const mg_grid* logits, const int32_t* target, float* logprob, float* loss,
                            mg_grid* dlogits, float gscale) {
  if (!ctx || !logits || !target) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, logits->H == 1 && logits->W == 1, MG_ERR_SHAPE, "nll: logits must be N x 1 x 1 x C");
  mg_sum* acc = loss ? mg_ctx_sum_scratch(ctx) : nullptr;
  MG_REQUIRE(ctx, !loss || acc, MG_ERR_CUDA, "nll: scratch allocation failed");
  MG_DISPATCH(ctx, nll_kernel<T><<<logits->N, 256, 0, ctx->stream>>>((const T*)logits->data, logits->C, logits->Cp, target, logprob, acc,
                                                                    dlogits ? (T*)dlogits->data : nullptr, dlogits ? dlogits->Cp : 0,
                                                                    gscale, logits->N););
  MG_CHECK_LAUNCH(ctx);
  if (loss) { loss_finalize_kernel<<<1, 1, 0, ctx->stream>>>(acc, loss); MG_CHECK_LAUNCH(ctx); }
  return MG_OK;
}

int mg_bce_forward_backward(mg_ctx* ctx, const mg_grid* x, const float* target_nchw, float* prob_nchw, float* loss,
                            mg_grid* dx, float gscale) {
  if (!ctx || !x || !target_nchw) return MG_ERR_INVALID_ARG;
  int64_t total = (int64_t)x->N * x->C * x->H * x->W;
  mg_sum* acc = loss ? mg_ctx_sum_scratch(ctx) : nullptr;
  MG_REQUIRE(ctx, !loss || acc, MG_ERR_CUDA, "bce: scratch allocation failed");
  MG_DISPATCH(ctx, bce_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*x), target_nchw, prob_nchw, acc,
                                                                      dx ? (T*)dx->data : nullptr, dx ? dx->Cp : 0, gscale););
  MG_CHECK_LAUNCH(ctx);
  if (loss) { loss_finalize_kernel<<<1, 1, 0, ctx->stream>>>(acc, loss); MG_CHECK_LAUNCH(ctx); }
  return MG_OK;
}

int mg_sgd_step(mg_ctx* ctx, float* w, const float* g, float* v, int64_t n, float lr, float momentum, float wd, int first) {
  if (!ctx || !w || !g || !v) return MG_ERR_INVALID_ARG;
  sgd_kernel<<<GRID1(n), EB, 0, ctx->stream>>>(w, g, v, n, lr, momentum, wd, first);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- module-level head ops
namespace {

// nn.LogSoftMax over the channel dim of an N x 1 x 1 x C grid, one block per sample
template <typename T>
__global__ void logsoftmax_fwd_kernel(const T* __restrict__ logits, int C, int ld, float* __restrict__ logprob) {
  int n = blockIdx.x;
  const T* row = logits + (size_t)n * ld;
  __shared__ float red[32];
  float m = -INFINITY;
  for (int c = threadIdx.x; c < C; c += blockDim.x) m = fmaxf(m, mg_ld(row + c));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = m;
  __syncthreads();
  m = red[0];
  for (int w = 1; w < blockDim.x / 32; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s += expf(mg_ld(row + c) - m);
  s = warp_sum(s);
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = s;
  __syncthreads();
  s = 0.f;
  for (int w = 0; w < blockDim.x / 32; ++w) s += red[w];
  float lse = m + logf(s);
  for (int c = threadIdx.x; c < C; c += blockDim.x) logprob[(size_t)n * C + c] = mg_ld(row + c) - lse;
}

// dlogits = grad_out - exp(logprob) * sum_c grad_out
template <typename T>
__global__ void logsoftmax_bwd_kernel(const float* __restrict__ logprob, const float* __restrict__ go, int C,
                                      T* __restrict__ dlogits, int ld) {
  int n = blockIdx.x;
  __shared__ float red[32];
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s += go[(size_t)n * C + c];
  s = warp_sum(s);
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = s;
  __syncthreads();
  s = 0.f;
  for (int w = 0; w < blockDim.x / 32; ++w) s += red[w];
  for (int c = threadIdx.x; c < ld; c += blockDim.x) {
    float v = 0.f;
    if (c < C) v = go[(size_t)n * C + c] - expf(logprob[(size_t)n * C + c]) * s;
    mg_st(dlogits + (size_t)n * ld + c, v);
  }
}

__global__ void nll_criterion_kernel(const float* __restrict__ logprob, const int32_t* __restrict__ target, int N, int C,
                                     mg_sum* loss, float* grad_out, float gscale) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  if (i >= (int64_t)N * C) return;
  int c = i % C, n = i / C;
  bool hit = target[n] == c;
  if (grad_out) grad_out[i] = hit ? -gscale / (float)N : 0.f;
  if (hit && loss) mg_sum_add(loss, (double)(-logprob[i] / (float)N));
}

__global__ void bce_criterion_kernel(const float* __restrict__ prob, const float* __restrict__ target, int64_t count,
                                     mg_sum* loss, float* grad, float gscale) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  float l = 0.f;
  if (i < count) {
    const float eps = 1e-12f;
    float p = prob[i], t = target[i];
    l = -(logf(p + eps) * t + logf(1.f - p + eps) * (1.f - t)) / (float)count;
    if (grad) grad[i] = -gscale * (t - p) / ((1.f - p + eps) * (p + eps)) / (float)count;
  }
  l = warp_sum(l);
  if (loss && threadIdx.x % 32 == 0 && l != 0.f) mg_sum_add(loss, (double)l);
}

template <typename T>
__global__ void sigmoid_fwd_kernel(GridV<T> x, float* __restrict__ prob) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)x.N * x.C * x.H * x.W;
  if (i >= total) return;
  int xx = i % x.W; int64_t p = i / x.W;
  int y = p % x.H; p /= x.H; int c = p % x.C; int n = p / x.C;
  prob[i] = 1.f / (1.f + expf(-x.at(n, y, xx, c)));
}

template <typename T>
__global__ void sigmoid_bwd_kernel(const float* __restrict__ prob, const float* __restrict__ go, T* __restrict__ dx,
                                   int N, int C, int Cp, int H, int W) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  int64_t total = (int64_t)N * H * W * Cp;
  if (i >= total) return;
  int c = i % Cp; int64_t p = i / Cp;
  int x = p % W; p /= W; int y = p % H; int n = p / H;
  float v = 0.f;
  if (c < C) {
    size_t j = (((size_t)n * C + c) * H + y) * W + x;
    float pr = prob[j];
    v = go[j] * pr * (1.f - pr);
  }
  mg_st(dx + i, v);
}

}  // namespace

extern "C" {

int mg_logsoftmax_forward(mg_ctx* ctx, const mg_grid* logits, float* logprob) {
  if (!ctx || !logits || !logprob) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, logits->H == 1 && logits->W == 1, MG_ERR_SHAPE, "logsoftmax: logits must be N x 1 x 1 x C");
  MG_DISPATCH(ctx, logsoftmax_fwd_kernel<T><<<logits->N, 256, 0, ctx->stream>>>((const T*)logits->data, logits->C, logits->Cp, logprob););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_logsoftmax_backward(mg_ctx* ctx, const float* logprob, const float* grad_out, mg_grid* dlogits) {
  if (!ctx || !logprob || !grad_out || !dlogits) return MG_ERR_INVALID_ARG;
  MG_DISPATCH(ctx, logsoftmax_bwd_kernel<T><<<dlogits->N, 256, 0, ctx->stream>>>(logprob, grad_out, dlogits->C, (T*)dlogits->data, dlogits->Cp););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_nll_criterion(mg_ctx* ctx, const float* logprob, const int32_t* target, int32_t N, int32_t C, float* loss,
                     float* grad_out, float gscale) {
  if (!ctx || !logprob || !target || N < 1 || C < 1) return MG_ERR_INVALID_ARG;
  mg_sum* acc = loss ? mg_ctx_sum_scratch(ctx) : nullptr;
  MG_REQUIRE(ctx, !loss || acc, MG_ERR_CUDA, "nll_criterion: scratch allocation failed");
  nll_criterion_kernel<<<GRID1((int64_t)N * C), EB, 0, ctx->stream>>>(logprob, target, N, C, acc, grad_out, gscale);
  if (loss) { MG_CHECK_LAUNCH(ctx); loss_finalize_kernel<<<1, 1, 0, ctx->stream>>>(acc, loss); }
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_bce_criterion(mg_ctx* ctx, const float* prob, const float* target, int64_t count, float* loss, float* grad_prob,
                     float gscale) {
  if (!ctx || !prob || !target || count < 1) return MG_ERR_INVALID_ARG;
  mg_sum* acc = loss ? mg_ctx_sum_scratch(ctx) : nullptr;
  MG_REQUIRE(ctx, !loss || acc, MG_ERR_CUDA, "bce_criterion: scratch allocation failed");
  bce_criterion_kernel<<<GRID1(count), EB, 0, ctx->stream>>>(prob, target, count, acc, grad_prob, gscale);
  if (loss) { MG_CHECK_LAUNCH(ctx); loss_finalize_kernel<<<1, 1, 0, ctx->stream>>>(acc, loss); }
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_sigmoid_forward(mg_ctx* ctx, const mg_grid* x, float* prob_nchw) {
  if (!ctx || !x || !prob_nchw) return MG_ERR_INVALID_ARG;
  int64_t total = (int64_t)x->N * x->C * x->H * x->W;
  MG_DISPATCH(ctx, sigmoid_fwd_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(make_view<T>(*x), prob_nchw););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

int mg_sigmoid_backward(mg_ctx* ctx, const float* prob_nchw, const float* grad_out_nchw, mg_grid* dx) {
  if (!ctx || !prob_nchw || !grad_out_nchw || !dx) return MG_ERR_INVALID_ARG;
  int64_t total = (int64_t)dx->N * dx->H * dx->W * dx->Cp;
  MG_DISPATCH(ctx, sigmoid_bwd_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>(prob_nchw, grad_out_nchw, (T*)dx->data, dx->N, dx->C, dx->Cp, dx->H, dx->W););
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- 2x2 stride-2 up-convolution (U-MG) ----
// cudnn.SpatialFullConvolution(nIP, nOP, 2,2, 2,2, 0,0) of models/mnist-cluttered/unmg.lua:35-52:
// every input pixel owns its 2x2 output block, y[n,2y+dy,2x+dx,co] = b[co] + sum_ci x[n,y,x,ci] * w[ci][co][dy][dx].
// CUDA-core kernels (fp32 accumulate): the layer belongs to the config-5 comparator, not to the hot path.
namespace {

template <typename T>
__global__ void upconv_fwd_kernel(const T* __restrict__ x, int x_cp, int Cin, const float* __restrict__ w, const float* __restrict__ bias,
                                  T* __restrict__ y, int y_cp, int Cout, int N, int H, int W) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  const int64_t total = (int64_t)N * 2 * H * 2 * W * y_cp;
  if (i >= total) return;
  const int co = i % y_cp; int64_t q = i / y_cp;
  const int ox = q % (2 * W); q /= 2 * W; const int oy = q % (2 * H); const int n = q / (2 * H);
  float acc = 0.f;
  if (co < Cout) {
    acc = bias ? bias[co] : 0.f;
    const T* xp = x + (((size_t)n * H + (oy >> 1)) * W + (ox >> 1)) * x_cp;
    const float* wp = w + (size_t)co * 4 + (oy & 1) * 2 + (ox & 1);
    for (int ci = 0; ci < Cin; ++ci) acc = fmaf(mg_ld(xp + ci), wp[(size_t)ci * Cout * 4], acc);
  }
  mg_st(y + i, acc);
}

template <typename T>
__global__ void upconv_dgrad_kernel(const T* __restrict__ g, int g_cp, int Cout, const float* __restrict__ w, T* __restrict__ dx, int x_cp,
                                    int Cin, int N, int H, int W) {
  int64_t i = (int64_t)blockIdx.x * EB + threadIdx.x;
  const int64_t total = (int64_t)N * H * W * x_cp;
  if (i >= total) return;
  const int ci = i % x_cp; int64_t q = i / x_cp;
  const int x = q % W; q /= W; const int y = q % H; const int n = q / H;
  float acc = 0.f;
  if (ci < Cin)
    for (int d = 0; d < 4; ++d) {
      const T* gp = g + (((size_t)n * 2 * H + 2 * y + (d >> 1)) * 2 * W + 2 * x + (d & 1)) * g_cp;
      const float* wp = w + (size_t)ci * Cout * 4 + d;
      for (int co = 0; co < Cout; ++co) acc = fmaf(mg_ld(gp + co), wp[co * 4], acc);
    }
  mg_st(dx + i, acc);
}

// one block per (ci, co-tile of 64 x 4 positions = 256 threads), pixel range split over blockIdx.z
template <typename T>
__global__ void __launch_bounds__(256) upconv_wgrad_kernel(const T* __restrict__ x, int x_cp, const T* __restrict__ g, int g_cp, float* partial,
                                                           int Cin, int Cout, int N, int H, int W, int64_t pix_per_z) {
  const int ci = blockIdx.x;
  const int co = blockIdx.y * 64 + (threadIdx.x >> 2), d = threadIdx.x & 3;
  const int64_t P = (int64_t)N * H * W;
  const int64_t p0 = (int64_t)blockIdx.z * pix_per_z, p1 = min(P, p0 + pix_per_z);
  if (co >= Cout) return;
  float acc = 0.f;
  for (int64_t p = p0; p < p1; ++p) {
    const int xx = p % W; const int64_t q = p / W; const int yy = q % H; const int n = q / H;
    const float xv = mg_ld(x + p * x_cp + ci);
    acc = fmaf(xv, mg_ld(g + (((size_t)n * 2 * H + 2 * yy + (d >> 1)) * 2 * W + 2 * xx + (d & 1)) * g_cp + co), acc);
  }
  partial[((size_t)blockIdx.z * Cin * Cout + (size_t)ci * Cout + co) * 4 + d] = acc;   // per-split partial sums, added in a fixed order below
}

// dst[i] += gscale * sum_z partial[z][i], z in increasing order (no floating-point atomics)
__global__ void partial_reduce_kernel(const float* __restrict__ partial, int splits, int64_t plane, float* __restrict__ dst, float gscale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += partial[(size_t)z * plane + i];
  dst[i] += gscale * s;
}

}  // namespace

int simt_dbias(mg_ctx* ctx, const mg_grid* g, int Cout, float* dbias, float gscale);

extern "C" {

int mg_upconv2x2_forward(mg_ctx* ctx, const mg_grid* x, const float* w, const float* bias, mg_grid* y, mg_sum* bn_sums) {
  if (!ctx || !x || !w || !y) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, y->H == 2 * x->H && y->W == 2 * x->W && y->N == x->N && !x->scale, MG_ERR_SHAPE, "upconv: y must be 2x the size of x");
  {   // bf16: one 1x1 tensor-core convolution to 4 * Cout channels + depth-to-space (upconv_tc.cu)
    const int rc = upconv_tc_forward(ctx, x, w, bias, y);
    if (rc > 0) return rc;
    if (rc == 0) return bn_sums ? mg_bn_stats(ctx, y, bn_sums) : MG_OK;
  }
  const int64_t total = (int64_t)y->N * y->H * y->W * y->Cp;
  MG_DISPATCH(ctx, upconv_fwd_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>((const T*)x->data, x->Cp, x->C, w, bias, (T*)y->data, y->Cp, y->C,
                                                                             x->N, x->H, x->W););
  MG_CHECK_LAUNCH(ctx);
  if (bn_sums) return mg_bn_stats(ctx, y, bn_sums);
  return MG_OK;
}

int mg_upconv2x2_backward(mg_ctx* ctx, const mg_grid* x, const float* w, const mg_grid* g, mg_grid* dx, float* dw, float* dbias,
                          float gscale) {
  if (!ctx || !x || !w || !g) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, g->H == 2 * x->H && g->W == 2 * x->W && g->N == x->N, MG_ERR_SHAPE, "upconv backward: g must be 2x the size of x");
  {
    const int rc = upconv_tc_backward(ctx, x, w, g, dx, dw, dbias, gscale);
    if (rc >= 0) return rc;
  }
  if (dx) {
    const int64_t total = (int64_t)x->N * x->H * x->W * dx->Cp;
    MG_DISPATCH(ctx, upconv_dgrad_kernel<T><<<GRID1(total), EB, 0, ctx->stream>>>((const T*)g->data, g->Cp, g->C, w, (T*)dx->data, dx->Cp, x->C,
                                                                                 x->N, x->H, x->W););
    MG_CHECK_LAUNCH(ctx);
  }
  if (dw) {
    const int64_t P = (int64_t)x->N * x->H * x->W;
    const int gy = (int)mg_cdiv(g->C, 64);
    int64_t z = std::max<int64_t>(1, std::min<int64_t>(mg_cdiv(P, 256), mg_cdiv((int64_t)ctx->num_sms * 8, (int64_t)x->C * gy)));
    const int64_t ppz = mg_cdiv(P, z);
    z = mg_cdiv(P, ppz);
    dim3 grid((unsigned)x->C, (unsigned)gy, (unsigned)z);
    const int64_t plane = (int64_t)x->C * g->C * 4;
    void* ws = nullptr;
    const int rcw = mg_ctx_workspace(ctx, (size_t)z * plane * sizeof(float), &ws);
    if (rcw) return rcw;
    MG_DISPATCH(ctx, upconv_wgrad_kernel<T><<<grid, 256, 0, ctx->stream>>>((const T*)x->data, x->Cp, (const T*)g->data, g->Cp, (float*)ws, x->C, g->C, x->N,
                                                                          x->H, x->W, ppz););
    MG_CHECK_LAUNCH(ctx);
    partial_reduce_kernel<<<(unsigned)mg_cdiv(plane, 256), 256, 0, ctx->stream>>>((const float*)ws, (int)z, plane, dw, gscale);
    MG_CHECK_LAUNCH(ctx);
  }
  if (dbias) return simt_dbias(ctx, g, g->C, dbias, gscale);
  return MG_OK;
}

}  // extern "C"
