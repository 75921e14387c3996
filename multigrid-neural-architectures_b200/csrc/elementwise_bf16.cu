// bf16 fast paths of the HBM-bound passes: every thread moves 8 channels (16 bytes) of a pixel
// -- or of a 2x2 pixel block when the pass pools, routes through an arg-max or sums an up-sampled
// gradient -- so each byte of every tensor is read once per pass with 128-bit coalesced accesses.
// Same arithmetic, expression for expression, as the generic kernels in elementwise.cu (which
// remain the fp32 path and the fallback for unaligned channel offsets).
#include "common.cuh"
#include <algorithm>

namespace {

typedef __nv_bfloat16 bf16;

struct V8 { float v[8]; };

// (a, b, c, d) with i = ((a * nb + b) * nc + c) * nd + d.  Work items of these passes are far below 2^32, where the four
// divisions are 32-bit (a 64-bit division is ~100 instructions -- more than the rest of a thread's work in the apply pass).
__device__ __forceinline__ void split4(int64_t i, int nb, int nc, int nd, int& a, int& b, int& c, int& d) {
  if (i < ((int64_t)1 << 32)) {
    uint32_t q = (uint32_t)i, t;
    t = q / (uint32_t)nd; d = (int)(q - t * (uint32_t)nd); q = t;
    t = q / (uint32_t)nc; c = (int)(q - t * (uint32_t)nc); q = t;
    t = q / (uint32_t)nb; b = (int)(q - t * (uint32_t)nb); a = (int)t;
  } else {
    int64_t q = i;
    d = (int)(q % nd); q /= nd; c = (int)(q % nc); q /= nc; b = (int)(q % nb); a = (int)(q / nb);
  }
}

// division by a run-time constant as multiply-high + shift (valid for dividends < 2^31): the index decode of the streaming
// passes was ~400 of their ~1000 instructions per thread with emulated divisions (ncu: issue slots 63-66 % busy)
struct FastDiv { uint32_t mul, shift, d; };
static inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f; f.d = d; f.mul = 0; f.shift = 0;
  if (d > 1) {
    uint32_t lg = 0;
    while ((1ull << lg) < d) ++lg;
    const uint32_t p = 31 + lg;
    f.mul = (uint32_t)(((1ull << p) + d - 1) / d);
    f.shift = p - 32;
  }
  return f;
}
__device__ __forceinline__ uint32_t fd_div(uint32_t n, const FastDiv& f) { return f.d == 1 ? n : (__umulhi(n, f.mul) >> f.shift); }

__device__ __forceinline__ V8 ld8(const bf16* p) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  V8 r;
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    r.v[2 * i] = __uint_as_float(w[i] << 16);
    r.v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
  return r;
}
__device__ __forceinline__ uint4 pack8(const V8& a) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a.v[2 * i], a.v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&t);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ V8 unpack8(const uint4& u) {
  V8 r;
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    r.v[2 * i] = __uint_as_float(w[i] << 16);
    r.v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
  return r;
}
__device__ __forceinline__ void ldf8(const float* p, float (&o)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}

// per-block reduction of per-thread channel sums into the global sums: fixed order inside the block (no floating-point
// atomics), deterministic integer accumulation across blocks (mg_sum).  Threads of a block own vector column
// (tid % V) and pixel lane (tid / V); V*8 <= 4096 channels.  sh: [2][lanes * V * 8] floats, lanes = blockDim.x / V.
__device__ __forceinline__ void block_channel_sums(const float (&a)[8], const float (&b)[8], int vc, int V, int C, bool active,
                                                   mg_sum* sums, float* sh) {
  const int lanes = blockDim.x / V, lane = threadIdx.x / V;
  const int plane = lanes * V * 8;
  if (active) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { sh[(lane * V + vc) * 8 + e] = a[e]; sh[plane + (lane * V + vc) * 8 + e] = b[e]; }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < V * 8; c += blockDim.x)
    if (c < C) {
      float sa = 0.f, sb = 0.f;
      for (int l = 0; l < lanes; ++l) { sa += sh[l * V * 8 + c]; sb += sh[plane + l * V * 8 + c]; }
      mg_sum_add(sums + c, (double)sa);
      mg_sum_add(sums + C + c, (double)sb);
    }
}

// ---------------------------------------------------------------- apply (BN + shortcut + ReLU [+ pool]) ----
struct ApplyP {
  const bf16* z; int z_cp; const float* scale; const float* shift; int z_relu;
  const bf16* s; int s_cp;      // shortcut or null; channels >= s_cp contribute nothing
  int relu;
  bf16* out; int o_cp;
  bf16* pooled; int p_cp;       // or null
  int N, H, W, C, Hp, Wp;
  // fused BatchNorm finalisation (bn != 0): scale / shift are derived in-kernel from the fp64 sums (training) or the
  // running statistics (evaluation) -- expression for expression bn_finalize_kernel -- and block 0 writes the
  // module state (running statistics, saved mean / invstd, scale / shift)
  int bn, training;
  const mg_sum* sums; int64_t count;
  const float* gamma; const float* beta; float* rmean; float* rvar; float eps, momentum;
  float* smean; float* sinvstd; float* scale_out; float* shift_out;
  FastDiv fd_v, fd_wp, fd_hp;   // index decode (items and pixels < 2^31: checked by the launcher)
  double inv_count, unbias;     // 1 / count, count / (count - 1)
};

// BatchNorm finalisation of the apply pass, per CTA (expression for expression bn_finalize_kernel).  Not inlined: its fp64
// arithmetic would otherwise set the register count of the streaming body (64 instead of 40 registers per thread).
__device__ __forceinline__ void apply_bn_prologue(const ApplyP& p, float* s_aff) {
  for (int c = threadIdx.x; c < p.z_cp; c += blockDim.x) {
    float scv = 0.f, shv = 0.f, mv = 0.f, iv = 0.f;
    if (c < p.C) {
      double mean, var;
      if (p.training) {
        // reciprocal of the count and the unbiasing factor come from the host as doubles, the inverse standard deviation from
        // rsqrt: no fp64 division / square root routine (each ~100 instructions, executed by every CTA of the pass)
        mean = mg_sum_get(p.sums[c]) * p.inv_count;
        var = mg_sum_get(p.sums[p.C + c]) * p.inv_count - mean * mean;   // biased
        if (var < 0) var = 0;
        if (p.rmean && blockIdx.x == 0) {
          const double unb = var * p.unbias;
          p.rmean[c] = (float)((1.0 - p.momentum) * p.rmean[c] + p.momentum * mean);
          p.rvar[c] = (float)((1.0 - p.momentum) * p.rvar[c] + p.momentum * unb);
        }
      } else {
        mean = p.rmean[c]; var = p.rvar[c];
      }
      const double invstd = rsqrt(var + (double)p.eps);
      const float g = p.gamma ? p.gamma[c] : 1.f, b = p.beta ? p.beta[c] : 0.f;
      scv = (float)(g * invstd);
      shv = (float)(b - g * invstd * mean);
      mv = (float)mean; iv = (float)invstd;
    }
    s_aff[c] = scv; s_aff[p.z_cp + c] = shv;
    if (blockIdx.x == 0) {
      p.scale_out[c] = scv; p.shift_out[c] = shv;
      if (p.smean) { p.smean[c] = mv; p.sinvstd[c] = iv; }
    }
  }
}

__global__ void __launch_bounds__(256, 3) apply_bf16_kernel(const __grid_constant__ ApplyP p) {
  pdl_launch();
  pdl_wait();
  extern __shared__ float s_aff[];   // [2][z_cp] when bn
  if (p.bn) {
    apply_bn_prologue(p, s_aff);
    __syncthreads();
  }
  const uint32_t V = (uint32_t)p.o_cp >> 3;
  const uint32_t total = (uint32_t)p.N * p.Hp * p.Wp * V;
  // grid-stride loop: large tensors run on ~6 CTAs per SM, so the BatchNorm prologue above (fp64 division / square root: ~400
  // instructions per thread) is paid once per several blocks instead of once per block
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
  uint32_t q = fd_div(i, p.fd_v);
  const uint32_t vc = i - q * V;
  uint32_t t = fd_div(q, p.fd_wp);
  const uint32_t px = q - t * (uint32_t)p.Wp;
  const uint32_t n = fd_div(t, p.fd_hp);
  const uint32_t py = t - n * (uint32_t)p.Hp;
  const int c0 = (int)vc * 8;
  float sc[8], sh[8];
  const bool has_aff = p.bn || p.scale != nullptr;
  if (p.bn) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { sc[e] = s_aff[c0 + e]; sh[e] = s_aff[p.z_cp + c0 + e]; }
  } else if (has_aff) { ldf8(p.scale + c0, sc); ldf8(p.shift + c0, sh); }
  const bool has_s = p.s != nullptr && c0 < p.s_cp;
  // every load of the 2x2 block is issued before the first use (the stores below may alias z as far as the compiler knows, so
  // it would otherwise order load - store - load: eight dependent round trips per thread instead of one).  Pixels outside the
  // grid re-read pixel 0 of the block (always valid) and are dropped at the store.
  const uint32_t y0 = 2 * py, x0 = 2 * px;
  const bool okx = x0 + 1 < (uint32_t)p.W, oky = y0 + 1 < (uint32_t)p.H;
  const bool ok[4] = {true, okx, oky, okx && oky};
  const uint32_t pix0 = (n * (uint32_t)p.H + y0) * (uint32_t)p.W + x0;
  const uint32_t pix[4] = {pix0, pix0 + (okx ? 1u : 0u), pix0 + (oky ? (uint32_t)p.W : 0u), pix0 + (okx && oky ? (uint32_t)p.W + 1u : 0u)};
  uint4 zr[4], sr[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) zr[k] = *reinterpret_cast<const uint4*>(p.z + (size_t)pix[k] * p.z_cp + c0);
  if (has_s) {
#pragma unroll
    for (int k = 0; k < 4; ++k) sr[k] = *reinterpret_cast<const uint4*>(p.s + (size_t)pix[k] * p.s_cp + c0);
  }
  const bool ragged = c0 + 8 > p.C;          // the vector holds pad channels (stored as zeros)
  const bool zrelu = p.z_relu != 0, relu = p.relu != 0;
  // the pooled companion is the maximum of the STORED bf16 values: packed bf16x2 maxima (NaN-propagating like the scalar form)
  __nv_bfloat162 best[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) best[j] = __halves2bfloat162(__ushort_as_bfloat16((unsigned short)0xFF80), __ushort_as_bfloat16((unsigned short)0xFF80));
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (!ok[k]) continue;
    V8 v = unpack8(zr[k]);
    if (has_aff) {
#pragma unroll
      for (int e = 0; e < 8; ++e) { v.v[e] = fmaf(v.v[e], sc[e], sh[e]); if (zrelu) v.v[e] = fmaxf(v.v[e], 0.f); }   // = mg_xform
    }
    if (has_s) {
      const V8 sv = unpack8(sr[k]);
#pragma unroll
      for (int e = 0; e < 8; ++e) v.v[e] += sv.v[e];
    }
    if (relu) {
#pragma unroll
      for (int e = 0; e < 8; ++e) v.v[e] = fmaxf(v.v[e], 0.f);
    }
    if (ragged) {
#pragma unroll
      for (int e = 0; e < 8; ++e) if (c0 + e >= p.C) v.v[e] = 0.f;
    }
    const uint4 u = pack8(v);
    *reinterpret_cast<uint4*>(p.out + (size_t)pix[k] * p.o_cp + c0) = u;
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) best[j] = __hmax2_nan(best[j], *reinterpret_cast<const __nv_bfloat162*>(&w[j]));
  }
  if (p.pooled && c0 < p.p_cp) {
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = *reinterpret_cast<uint32_t*>(&best[j]);
    if (ragged) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (c0 + 2 * j >= p.C) w[j] &= 0xFFFF0000u;
        if (c0 + 2 * j + 1 >= p.C) w[j] &= 0x0000FFFFu;
      }
    }
    *reinterpret_cast<uint4*>(p.pooled + (size_t)((n * (uint32_t)p.Hp + py) * (uint32_t)p.Wp + px) * p.p_cp + c0) = make_uint4(w[0], w[1], w[2], w[3]);
  }
  }
}

// ---------------------------------------------------------------- BN statistics ----------
__global__ void __launch_bounds__(256) bn_stats_bf16_kernel(const bf16* __restrict__ y, int cp, int C, int64_t P, mg_sum* sums) {
  pdl_launch();
  pdl_wait();
  extern __shared__ float sh[];
  const int V = cp >> 3;
  // each CTA streams ONE contiguous pixel range (DRAM page locality); inside it the threads of a CTA form
  // `lanes` pixel lanes x V channel vectors and walk the range lane-strided
  const int lanes = blockDim.x / V;            // threads beyond lanes*V idle
  const int vc = threadIdx.x % V, lane = threadIdx.x / V;
  const int64_t per_cta = (P + gridDim.x - 1) / gridDim.x;
  const int64_t p_begin = (int64_t)blockIdx.x * per_cta, p_end = min(P, p_begin + per_cta);
  float a[8], b[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { a[e] = 0.f; b[e] = 0.f; }
  const bool active = lane < lanes;
  if (active) {
    int64_t pix = p_begin + lane;
    for (; pix + 3 * lanes < p_end; pix += 4 * lanes) {   // four independent 16-byte loads in flight per thread
      V8 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ld8(y + (pix + u * lanes) * cp + vc * 8);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int e = 0; e < 8; ++e) { a[e] += v[u].v[e]; b[e] = fmaf(v[u].v[e], v[u].v[e], b[e]); }
    }
    for (; pix < p_end; pix += lanes) {
      const V8 v = ld8(y + pix * cp + vc * 8);
#pragma unroll
      for (int e = 0; e < 8; ++e) { a[e] += v.v[e]; b[e] = fmaf(v.v[e], v.v[e], b[e]); }
    }
  }
  block_channel_sums(a, b, vc, V, C, active, sums, sh);
}

// ---------------------------------------------------------------- gradient combine ----------
struct CSrc { const bf16* g; const uint8_t* aux; int H, W, cp, c_off, mode; };
struct CombP {
  const bf16* x; int x_cp;       // activation tensor (ReLU mask, pool arg-max)
  const bf16* bnx; int bn_cp;    // raw conv output for the BatchNorm sums, or null
  int relu_mask;
  int n_src; CSrc src[MG_MAX_SRC];
  bf16* d; int d_cp;
  mg_sum* sums;
  int N, H, W, C, Hb, Wb;        // Hb = ceil(H/2): 2x2 blocks
  FastDiv fd_wb, fd_hb;          // combine_fast_kernel: index decode
  // frozen BatchNorm (combine_fast_kernel<.., true>): G = A * d with A = gamma * invstd_r derived per CTA; d is stored only when
  // p.d is set (a residual shortcut reads it)
  const float* fz_gamma; const float* fz_rvar; float fz_eps;
  bf16* g; int g_cp;
};

// NS >= 0: the number of sources and their modes (2 bits each in MODES) are compile-time constants, so the source loop
// unrolls, the mode branches fold and the compiler can issue the loads of ALL sources of a 2x2 block back to back
// (the pass is latency bound: bytes in flight per SM are what matters).  NS < 0: generic (run-time source list).
__device__ __forceinline__ V8 ldg8(const bf16* p) { return unpack8(__ldg(reinterpret_cast<const uint4*>(p))); }

template <int NS, int MODES>
__global__ void __launch_bounds__(256, NS < 0 ? 3 : 2) combine_bf16_kernel(const __grid_constant__ CombP p) {
  pdl_launch();
  pdl_wait();
  extern __shared__ float sh[];
  const int V = p.d_cp >> 3;
  const int lanes = blockDim.x / V;
  const int vc = threadIdx.x % V, lane = threadIdx.x / V;
  const int c0 = vc * 8;
  const int64_t nblocks = (int64_t)p.N * p.Hb * p.Wb;
  const int64_t per_cta = (nblocks + gridDim.x - 1) / gridDim.x;   // contiguous range of 2x2 blocks per CTA
  const int64_t b_begin = (int64_t)blockIdx.x * per_cta, b_end = min(nblocks, b_begin + per_cta);
  const bool active = lane < lanes;
  float sd[8], sdx[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { sd[e] = 0.f; sdx[e] = 0.f; }
  const int n_src = NS < 0 ? p.n_src : NS;
  bool need_x = p.relu_mask != 0;
#pragma unroll
  for (int s = 0; s < (NS < 0 ? MG_MAX_SRC : NS); ++s)
    if (s < n_src) need_x = need_x || (NS < 0 ? p.src[s].mode : ((MODES >> (2 * s)) & 3)) == MG_SEG_POOL;

  if (active)
    for (int64_t blk = b_begin + lane; blk < b_end; blk += lanes) {
      int n, by, bx, unused_;
      split4(blk, p.Hb, p.Wb, 1, n, by, bx, unused_);
      const int y0 = 2 * by, x0 = 2 * bx;
      const bool vy1 = y0 + 1 < p.H, vx1 = x0 + 1 < p.W;
      const bool valid[4] = {true, vx1, vy1, vy1 && vx1};
      int64_t pix[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) pix[k] = ((int64_t)n * p.H + y0 + (k >> 1)) * p.W + x0 + (k & 1);
      uint4 Xr[4];   // raw bf16 (4 registers each); unpacked where needed
#pragma unroll
      for (int k = 0; k < 4; ++k) Xr[k] = make_uint4(0, 0, 0, 0);
      if (need_x) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (valid[k]) Xr[k] = __ldg(reinterpret_cast<const uint4*>(p.x + pix[k] * p.x_cp + c0));
      }
      V8 acc[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[k].v[e] = 0.f;

#pragma unroll
      for (int s = 0; s < (NS < 0 ? MG_MAX_SRC : NS); ++s) {
        if (s >= n_src) break;
        const CSrc& S = p.src[s];
        const int mode = NS < 0 ? S.mode : ((MODES >> (2 * s)) & 3);
        if (mode == MG_SEG_SAME) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (valid[k]) {
              const V8 g = ldg8(S.g + pix[k] * S.cp + S.c_off + c0);
#pragma unroll
              for (int e = 0; e < 8; ++e) acc[k].v[e] += g.v[e];
            }
        } else if (mode == MG_SEG_UP) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (valid[k]) {
              const int y = y0 + (k >> 1), x = x0 + (k & 1);
              const bf16* gp = S.g + (((int64_t)n * S.H + 2 * y) * S.W + 2 * x) * S.cp + S.c_off + c0;
              const V8 g0 = ldg8(gp), g1 = ldg8(gp + S.cp), g2 = ldg8(gp + (int64_t)S.W * S.cp), g3 = ldg8(gp + (int64_t)S.W * S.cp + S.cp);
#pragma unroll
              for (int e = 0; e < 8; ++e) acc[k].v[e] += g0.v[e] + g1.v[e] + g2.v[e] + g3.v[e];
            }
        } else if (mode == MG_SEG_POOL) {
          // this 2x2 block is exactly one pooling window: route to the first maximum (row-major scan)
          const V8 g = ldg8(S.g + (((int64_t)n * S.H + by) * S.W + bx) * S.cp + S.c_off + c0);
          V8 X[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) X[k] = unpack8(Xr[k]);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float best = -INFINITY; int bi = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (valid[k]) { const float v = X[k].v[e]; if (v > best || v != v) { best = v; bi = k; } }
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (bi == k) acc[k].v[e] += g.v[e];
          }
        } else {
          // SpatialMaxPooling(3,3,2,2,1,1) of the stem: arg-max code (ky*3+kx) stored by the forward pass
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (valid[k]) {
              const int y = y0 + (k >> 1), x = x0 + (k & 1);
              const int oy0 = max(y / 2, 0), oy1 = min((y + 1) / 2, S.H - 1);
              const int ox0 = max(x / 2, 0), ox1 = min((x + 1) / 2, S.W - 1);
              for (int oy = oy0; oy <= oy1; ++oy)
                for (int ox = ox0; ox <= ox1; ++ox) {
                  const int64_t o = ((int64_t)n * S.H + oy) * S.W + ox;
                  const uint2 code = __ldg(reinterpret_cast<const uint2*>(S.aux + o * S.cp + S.c_off + c0));
                  const int want = (y - (2 * oy - 1)) * 3 + (x - (2 * ox - 1));
                  const V8 g = ldg8(S.g + o * S.cp + S.c_off + c0);
#pragma unroll
                  for (int e = 0; e < 8; ++e) {
                    const int cd = ((e < 4 ? code.x : code.y) >> (8 * (e & 3))) & 0xFF;
                    if (cd == want) acc[k].v[e] += g.v[e];
                  }
                }
            }
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (valid[k]) {
          const V8 xk = unpack8(Xr[k]);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            if (p.relu_mask && !(xk.v[e] > 0.f)) acc[k].v[e] = 0.f;
            if (c0 + e >= p.C) acc[k].v[e] = 0.f;
          }
          if (p.sums) {
            const V8 yr = ldg8(p.bnx + pix[k] * p.bn_cp + c0);
#pragma unroll
            for (int e = 0; e < 8; ++e) { sd[e] += acc[k].v[e]; sdx[e] = fmaf(acc[k].v[e], yr.v[e], sdx[e]); }
          }
          *reinterpret_cast<uint4*>(p.d + pix[k] * p.d_cp + c0) = pack8(acc[k]);
        }
    }
  if (p.sums) block_channel_sums(sd, sdx, vc, V, p.C, active, p.sums, sh);
}

// The specialised lists whose modes are same / pool / up only: all loads of a 2x2 block are issued as raw 16-byte registers
// before the first use (first the 16 of an up-sampled source, which are summed at once; then the activation, the raw
// BatchNorm input and every same / pool source together), so a thread has up to 17 independent loads in flight instead of a
// chain of dependent ones (the older form above reuses one destination register for consecutive loads and interleaves the
// BatchNorm-input loads with the stores: ~13 round trips per block).  Pixels outside the grid (odd H / W) re-read pixel 0 of
// the block and are dropped at the store.  Same arithmetic and summation order as combine_bf16_kernel.
//
// FROZEN: the tensor feeds a BatchNorm in evaluation mode, a fixed per-channel affine, so its backward is G = A * d with
// A = gamma * invstd_r (frozen_bn_invstd, as mg_bn_finalize derives it from the running variance).  The same pass writes G
// (and d only when p.d is set), still accumulating (sum d, sum d*y) for dgamma / dbeta (mg_bn_backward_frozen): no second pass
// over d and y.
// The frozen form keeps the batched loads of its 2x2 block AND the product with A live at once: at two CTAs per SM (128 registers)
// the longer source lists spill, so it runs one CTA per SM with the whole register budget.
template <int NS, int MODES, bool FROZEN>
__global__ void __launch_bounds__(256, FROZEN ? 1 : 2) combine_fast_kernel(const __grid_constant__ CombP p) {
  pdl_launch();
  pdl_wait();
  extern __shared__ float sh[];
  const int V = p.d_cp >> 3;
  const int lanes = blockDim.x / V;
  const int vc = threadIdx.x % V, lane = threadIdx.x / V;
  const int c0 = vc * 8;
  const uint32_t nblocks = (uint32_t)p.N * p.Hb * p.Wb;       // blocks and pixels < 2^31: checked by the launcher
  const uint32_t per_cta = (nblocks + gridDim.x - 1) / gridDim.x;
  const uint32_t b_begin = blockIdx.x * per_cta, b_end = min(nblocks, b_begin + per_cta);
  const bool active = lane < lanes;
  float sd[8], sdx[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { sd[e] = 0.f; sdx[e] = 0.f; }
  constexpr bool any_pool = ((MODES & 3) == 1 && NS > 0) || (((MODES >> 2) & 3) == 1 && NS > 1) || (((MODES >> 4) & 3) == 1 && NS > 2) ||
                            (((MODES >> 6) & 3) == 1 && NS > 3);
  const bool need_x = p.relu_mask == 1 || any_pool;   // relu_mask == 2: x is the POOLED tensor of the single mode-3 source (stem)
  const bool has_sums = p.sums != nullptr;
  float* s_a = sh + 2 * 256 * 8;   // FROZEN: A per channel, after the block_channel_sums staging (read at the store: no registers held)
  if (FROZEN) {
    for (int c = threadIdx.x; c < p.g_cp; c += blockDim.x)
      s_a[c] = c < p.C ? (float)((p.fz_gamma ? (double)p.fz_gamma[c] : 1.0) * frozen_bn_invstd(p.fz_rvar[c], p.fz_eps)) : 0.f;
    __syncthreads();
  }

  if (active)
    for (uint32_t blk = b_begin + lane; blk < b_end; blk += lanes) {
      const uint32_t tq = fd_div(blk, p.fd_wb);
      const int bx = (int)(blk - tq * (uint32_t)p.Wb);
      const int n = (int)fd_div(tq, p.fd_hb);
      const int by = (int)(tq - (uint32_t)n * (uint32_t)p.Hb);
      const int y0 = 2 * by, x0 = 2 * bx;
      const bool vy1 = y0 + 1 < p.H, vx1 = x0 + 1 < p.W;
      const bool valid[4] = {true, vx1, vy1, vy1 && vx1};
      const uint32_t pix0 = ((uint32_t)n * (uint32_t)p.H + (uint32_t)y0) * (uint32_t)p.W + (uint32_t)x0;
      const uint32_t pix[4] = {pix0, pix0 + (vx1 ? 1u : 0u), pix0 + (vy1 ? (uint32_t)p.W : 0u), pix0 + (vy1 && vx1 ? (uint32_t)p.W + 1u : 0u)};
      V8 acc[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[k].v[e] = 0.f;
      // ---- up-sampled sources: this tensor was up-sampled into the consumer, so each pixel collects a 2x2 block of g ----
#pragma unroll
      for (int s = 0; s < NS; ++s)
        if (((MODES >> (2 * s)) & 3) == MG_SEG_UP) {
          const CSrc& S = p.src[s];
          uint4 r[16];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int y = y0 + (valid[k] ? (k >> 1) : 0), x = x0 + (valid[k] ? (k & 1) : 0);
            const bf16* gp = S.g + (size_t)(((uint32_t)n * (uint32_t)S.H + 2u * (uint32_t)y) * (uint32_t)S.W + 2u * (uint32_t)x) * S.cp + S.c_off + c0;
            r[4 * k] = __ldg(reinterpret_cast<const uint4*>(gp));
            r[4 * k + 1] = __ldg(reinterpret_cast<const uint4*>(gp + S.cp));
            r[4 * k + 2] = __ldg(reinterpret_cast<const uint4*>(gp + (int64_t)S.W * S.cp));
            r[4 * k + 3] = __ldg(reinterpret_cast<const uint4*>(gp + (int64_t)S.W * S.cp + S.cp));
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const V8 g0 = unpack8(r[4 * k]), g1 = unpack8(r[4 * k + 1]), g2 = unpack8(r[4 * k + 2]), g3 = unpack8(r[4 * k + 3]);
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[k].v[e] += g0.v[e] + g1.v[e] + g2.v[e] + g3.v[e];
          }
        }
      // ---- everything else, raw ----
      uint4 Xr[4], Yr[4], Gr[NS > 0 ? NS : 1][4];
      uint2 Cd[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { Xr[k] = make_uint4(0, 0, 0, 0); Yr[k] = make_uint4(0, 0, 0, 0); }
      if (need_x) {
#pragma unroll
        for (int k = 0; k < 4; ++k) Xr[k] = __ldg(reinterpret_cast<const uint4*>(p.x + (size_t)pix[k] * p.x_cp + c0));
      }
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const CSrc& S = p.src[s];
        const int mode = (MODES >> (2 * s)) & 3;
        if (mode == MG_SEG_SAME) {
#pragma unroll
          for (int k = 0; k < 4; ++k) Gr[s][k] = __ldg(reinterpret_cast<const uint4*>(S.g + (size_t)pix[k] * S.cp + S.c_off + c0));
        } else if (mode == MG_SEG_POOL) {
          Gr[s][0] = __ldg(reinterpret_cast<const uint4*>(S.g + (size_t)(((uint32_t)n * (uint32_t)S.H + (uint32_t)by) * (uint32_t)S.W + (uint32_t)bx) * S.cp + S.c_off + c0));
        } else if (mode == 3) {
          // SpatialMaxPooling(3,3,2,2,1,1) of the stem: the 2x2 block lies in the four windows (by + wy, bx + wx); window w of the
          // block is loaded once (gradient + arg-max codes) instead of once per pixel it covers
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int oy = min(by + (w >> 1), S.H - 1), ox = min(bx + (w & 1), S.W - 1);
            const size_t o = (size_t)(((uint32_t)n * (uint32_t)S.H + (uint32_t)oy) * (uint32_t)S.W + (uint32_t)ox);
            Gr[s][w] = __ldg(reinterpret_cast<const uint4*>(S.g + o * S.cp + S.c_off + c0));
            Cd[w] = __ldg(reinterpret_cast<const uint2*>(S.aux + o * S.cp + S.c_off + c0));
            // the activation was never stored (mg_bn_relu_pool3_forward): its ReLU mask at an arg-max is the sign of the pooled value
            if (p.relu_mask == 2) Xr[w] = __ldg(reinterpret_cast<const uint4*>(p.x + o * p.x_cp + c0));
          }
        }
      }
      if (has_sums) {
#pragma unroll
        for (int k = 0; k < 4; ++k) Yr[k] = __ldg(reinterpret_cast<const uint4*>(p.bnx + (size_t)pix[k] * p.bn_cp + c0));
      }
      // ---- accumulate: up-sampled sources first (above), then the others in list order.  The order is a property of the
      // source-mode list alone (never of the launch, the lane or the run), so results stay reproducible; against the generic
      // kernel the fp32 sum of the <= 4 sources may differ in its last bit for lists with an up-sampled source ----
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int mode = (MODES >> (2 * s)) & 3;
        if (mode == MG_SEG_SAME) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const V8 g = unpack8(Gr[s][k]);
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[k].v[e] += g.v[e];
          }
        } else if (mode == MG_SEG_POOL) {
          const V8 g = unpack8(Gr[s][0]);
          V8 X[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) X[k] = unpack8(Xr[k]);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float best = -INFINITY; int bi = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (valid[k]) { const float v = X[k].v[e]; if (v > best || v != v) { best = v; bi = k; } }
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (bi == k) acc[k].v[e] += g.v[e];
          }
        } else if (mode == 3) {
          const CSrc& S = p.src[s];
          // pixel (dy, dx) of the block lies in window (wy, wx) iff (wy == 0 || dy == 1) && (wx == 0 || dx == 1), at tap
          // (dy + 1 - 2 wy, dx + 1 - 2 wx); windows in (oy, ox) order as the generic kernel visits them
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int wy = w >> 1, wx = w & 1;
            if (by + wy >= S.H || bx + wx >= S.W) continue;
            V8 g = unpack8(Gr[s][w]);
            if (p.relu_mask == 2) {
              const V8 pw = unpack8(Xr[w]);
#pragma unroll
              for (int e = 0; e < 8; ++e) if (!(pw.v[e] > 0.f)) g.v[e] = 0.f;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int dy = k >> 1, dx = k & 1;
              if ((wy == 1 && dy == 0) || (wx == 1 && dx == 0)) continue;
              const int want = (dy + 1 - 2 * wy) * 3 + (dx + 1 - 2 * wx);
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int cd = ((e < 4 ? Cd[w].x : Cd[w].y) >> (8 * (e & 3))) & 0xFF;
                if (cd == want) acc[k].v[e] += g.v[e];
              }
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (valid[k]) {
          const V8 xk = unpack8(Xr[k]);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            if (p.relu_mask == 1 && !(xk.v[e] > 0.f)) acc[k].v[e] = 0.f;
            if (c0 + e >= p.C) acc[k].v[e] = 0.f;
          }
          if (has_sums) {
            const V8 yr = unpack8(Yr[k]);
#pragma unroll
            for (int e = 0; e < 8; ++e) { sd[e] += acc[k].v[e]; sdx[e] = fmaf(acc[k].v[e], yr.v[e], sdx[e]); }
          }
          if (!FROZEN || p.d) *reinterpret_cast<uint4*>(p.d + (size_t)pix[k] * p.d_cp + c0) = pack8(acc[k]);
          if (FROZEN) {
            V8 gk;
#pragma unroll
            for (int e = 0; e < 8; ++e) gk.v[e] = s_a[c0 + e] * acc[k].v[e];
            *reinterpret_cast<uint4*>(p.g + (size_t)pix[k] * p.g_cp + c0) = pack8(gk);
          }
        }
    }
  if (p.sums) block_channel_sums(sd, sdx, vc, V, p.C, active, p.sums, sh);
}

// ---------------------------------------------------------------- BN backward apply ----------
// G = A*D + B*y + C per channel.  The gradBias of the convolution that produced y (accGradParameters: sum over pixels of
// G) needs no pass over G: sum G = A * sum d + B * sum y + C * n, all known from the sums -- and identically zero in exact
// arithmetic (training-mode BatchNorm removes the mean), i.e. pure rounding noise in the reference too.  Block 0 adds the
// fp64 evaluation of that expression; nothing is reduced with floating-point atomics.
struct BnBwdP {   // coefficients derived in-kernel (bn_bwd_coef_kernel, expression for expression); block 0 accumulates dgamma / dbeta
  const mg_sum* sums; int64_t count;
  const float* gamma; const float* mean; const float* invstd;
  float* dgamma; float* dbeta;
  double inv_count;
};

__global__ void __launch_bounds__(256, 3) bn_bwd_apply_bf16_kernel(const bf16* __restrict__ xraw, int x_cp, const bf16* d, int d_cp, bf16* out,
                                                                int o_cp, int C, int64_t P, BnBwdP bp,
                                                                float* dbias, float gscale) {
  pdl_launch();
  pdl_wait();
  extern __shared__ float sh[];   // [3][V*8] coefficients
  const int V = o_cp >> 3;
  float* s_coef = sh;
  for (int c = threadIdx.x; c < V * 8; c += blockDim.x) {
    float A = 0.f, B = 0.f, Cc = 0.f;
    if (c < C) {
      const double sd = mg_sum_get(bp.sums[c]), sdx = mg_sum_get(bp.sums[C + c]);
      const double mu = bp.mean[c], is = bp.invstd[c], g = bp.gamma ? bp.gamma[c] : 1.0;
      const double n = (double)bp.count, rn = bp.inv_count;   // reciprocal from the host: no fp64 division routine per CTA
      const BnTrainTerms t = bn_train_terms<true>(sd, sdx, mu, is, g, n, rn);
      if (blockIdx.x == 0) bn_train_param_grad(t, sd, mu, n, c, bp.dgamma, bp.dbeta, dbias, gscale);
      A = (float)t.Ad; B = (float)t.Bd; Cc = (float)t.Cd;
    }
    s_coef[c] = A; s_coef[V * 8 + c] = B; s_coef[2 * V * 8 + c] = Cc;
  }
  __syncthreads();
  const int lanes = blockDim.x / V;
  const int vc = threadIdx.x % V, lane = threadIdx.x / V;
  const int c0 = vc * 8;
  const bool active = lane < lanes;
  const int64_t per_cta = (P + gridDim.x - 1) / gridDim.x;      // contiguous pixel range per CTA
  const int64_t p_begin = (int64_t)blockIdx.x * per_cta, p_end = min(P, p_begin + per_cta);
  if (active) {
    float A[8], B[8], Cc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { A[e] = s_coef[c0 + e]; B[e] = s_coef[V * 8 + c0 + e]; Cc[e] = s_coef[2 * V * 8 + c0 + e]; }
    for (int64_t pix0 = p_begin + lane; pix0 < p_end; pix0 += 4 * lanes) {
      uint4 dr[4], xr[4];   // raw bf16, unpacked at use
#pragma unroll
      for (int u = 0; u < 4; ++u) {   // eight independent 16-byte loads in flight per thread
        const int64_t pix = pix0 + u * lanes;
        dr[u] = make_uint4(0, 0, 0, 0); xr[u] = make_uint4(0, 0, 0, 0);
        if (pix < p_end) {
          dr[u] = *reinterpret_cast<const uint4*>(d + pix * d_cp + c0);   // d may alias out: no read-only path
          xr[u] = __ldg(reinterpret_cast<const uint4*>(xraw + pix * x_cp + c0));
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t pix = pix0 + u * lanes;
        if (pix < p_end) {
          const V8 dv = unpack8(dr[u]), xv = unpack8(xr[u]);
          V8 o;
#pragma unroll
          for (int e = 0; e < 8; ++e) o.v[e] = (c0 + e < C) ? fmaf(A[e], dv.v[e], fmaf(B[e], xv.v[e], Cc[e])) : 0.f;
          *reinterpret_cast<uint4*>(out + pix * o_cp + c0) = pack8(o);
        }
      }
    }
  }
}

// ---------------------------------------------------------------- stem max-pool with arg-max codes ----------
__global__ void __launch_bounds__(256) pool3_bf16_kernel(const bf16* __restrict__ in, int H, int W, int cp, int C, bf16* __restrict__ out,
                                                         uint8_t* __restrict__ code, int Ho, int Wo, int N) {
  const int V = cp >> 3;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)N * Ho * Wo * V) return;
  int n, oy, ox, vc;
  split4(i, Ho, Wo, V, n, oy, ox, vc);
  const int c0 = vc * 8;
  float best[8]; int bc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { best[e] = -INFINITY; bc[e] = -1; }
  // the nine taps are loaded before the first comparison (taps outside the image re-read a clamped pixel and are skipped)
  uint4 r[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int y = min(max(2 * oy - 1 + t / 3, 0), H - 1), x = min(max(2 * ox - 1 + t % 3, 0), W - 1);
    r[t] = __ldg(reinterpret_cast<const uint4*>(in + (((int64_t)n * H + y) * W + x) * cp + c0));
  }
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int y = 2 * oy - 1 + t / 3, x = 2 * ox - 1 + t % 3;
    if (y < 0 || y >= H || x < 0 || x >= W) continue;
    const V8 v = unpack8(r[t]);
#pragma unroll
    for (int e = 0; e < 8; ++e)
      if (v.v[e] > best[e] || v.v[e] != v.v[e] || bc[e] < 0) { best[e] = v.v[e]; bc[e] = t; }
  }
  V8 b;
#pragma unroll
  for (int e = 0; e < 8; ++e) b.v[e] = (c0 + e < C) ? best[e] : 0.f;
  const int64_t o = ((int64_t)n * Ho + oy) * Wo + ox;
  *reinterpret_cast<uint4*>(out + o * cp + c0) = pack8(b);
  if (code) {
    uint2 cd;
    cd.x = (uint32_t)bc[0] | ((uint32_t)bc[1] << 8) | ((uint32_t)bc[2] << 16) | ((uint32_t)bc[3] << 24);
    cd.y = (uint32_t)bc[4] | ((uint32_t)bc[5] << 8) | ((uint32_t)bc[6] << 16) | ((uint32_t)bc[7] << 24);
    *reinterpret_cast<uint2*>(code + o * cp + c0) = cd;
  }
}

// ---------------------------------------------------------------- stem: BN + ReLU + 3x3 / stride-2 max-pool in one pass ----------
// SpatialBatchNormalization -> ReLU -> SpatialMaxPooling(3,3,2,2,1,1) of the ImageNet stem (models/ilsvrc/rnmg.lua:181-183) without
// the full-resolution activation: one thread = one pooled pixel x 8 channels reads its 3x3 window of the raw conv output, applies
// the (fused, apply_bn_prologue) BatchNorm affine and the ReLU, rounds to bf16 exactly where the two-pass form stores, and keeps
// the first maximum + its tap code.  The activation is only ever consumed by the pool, and backward needs it only for the ReLU
// mask AT the arg-max, where it equals the pooled value (combine: relu_mask = 2) -- so it never exists in HBM: per step 0.54 GB not
// written and 1.1 GB not read back.
__global__ void __launch_bounds__(256, 3) bn_relu_pool3_bf16_kernel(const __grid_constant__ ApplyP p, uint8_t* __restrict__ code, int Ho, int Wo) {
  pdl_launch();
  pdl_wait();
  extern __shared__ float s_aff[];   // [2][z_cp]
  apply_bn_prologue(p, s_aff);
  __syncthreads();
  const uint32_t V = (uint32_t)p.o_cp >> 3;
  const uint32_t total = (uint32_t)p.N * Ho * Wo * V;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    uint32_t q = fd_div(i, p.fd_v);
    const uint32_t vc = i - q * V;
    uint32_t t = fd_div(q, p.fd_wp);                 // fd_wp / fd_hp hold Wo / Ho here
    const int ox = (int)(q - t * (uint32_t)Wo);
    const uint32_t n = fd_div(t, p.fd_hp);
    const int oy = (int)(t - n * (uint32_t)Ho);
    const int c0 = (int)vc * 8;
    float sc[8], sh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { sc[e] = s_aff[c0 + e]; sh[e] = s_aff[p.z_cp + c0 + e]; }
    uint4 r[9];
#pragma unroll
    for (int tp = 0; tp < 9; ++tp) {
      const int y = min(max(2 * oy - 1 + tp / 3, 0), p.H - 1), x = min(max(2 * ox - 1 + tp % 3, 0), p.W - 1);
      r[tp] = __ldg(reinterpret_cast<const uint4*>(p.z + (size_t)((n * (uint32_t)p.H + (uint32_t)y) * (uint32_t)p.W + (uint32_t)x) * p.z_cp + c0));
    }
    // arg-max on packed bf16 pairs (the kernel is issue bound: 9 taps x 8 channels per thread): strictly-greater keeps the FIRST
    // maximum like the scalar pool (values are >= 0 after the ReLU, so the first valid tap always beats the -inf start)
    __nv_bfloat162 best[4];
    uint32_t bc[4];                 // two 16-bit tap codes per register
    const __nv_bfloat162 ninf = __halves2bfloat162(__ushort_as_bfloat16((unsigned short)0xFF80), __ushort_as_bfloat16((unsigned short)0xFF80));
#pragma unroll
    for (int j = 0; j < 4; ++j) { best[j] = ninf; bc[j] = 0; }
    const bool ragged = c0 + 8 > p.C;
#pragma unroll
    for (int tp = 0; tp < 9; ++tp) {
      const int y = 2 * oy - 1 + tp / 3, x = 2 * ox - 1 + tp % 3;
      if (y < 0 || y >= p.H || x < 0 || x >= p.W) continue;
      const V8 v = unpack8(r[tp]);
      V8 a;
#pragma unroll
      for (int e = 0; e < 8; ++e) a.v[e] = fmaxf(fmaf(v.v[e], sc[e], sh[e]), 0.f);   // = mg_xform + ReLU
      if (ragged) {
#pragma unroll
        for (int e = 0; e < 8; ++e) if (c0 + e >= p.C) a.v[e] = 0.f;                  // pad channels zero
      }
      const uint4 u = pack8(a);                                                        // what the apply pass would have stored
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
      const uint32_t tp2 = (uint32_t)tp * 0x00010001u;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const __nv_bfloat162 ab = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
        const uint32_t m = __hgt2_mask(ab, best[j]);                                   // 0xFFFF per half where ab > best
        best[j] = __hmax2(best[j], ab);
        bc[j] = (tp2 & m) | (bc[j] & ~m);
      }
    }
    const size_t o = (size_t)((n * (uint32_t)Ho + (uint32_t)oy) * (uint32_t)Wo + (uint32_t)ox);
    *reinterpret_cast<uint4*>(p.out + o * p.o_cp + c0) = make_uint4(*reinterpret_cast<uint32_t*>(&best[0]), *reinterpret_cast<uint32_t*>(&best[1]),
                                                                     *reinterpret_cast<uint32_t*>(&best[2]), *reinterpret_cast<uint32_t*>(&best[3]));
    uint2 cd;   // byte e = code of channel c0 + e: register j holds channels 2j (low half) and 2j + 1 (high half)
    cd.x = (bc[0] & 0xFF) | ((bc[0] >> 16 & 0xFF) << 8) | ((bc[1] & 0xFF) << 16) | ((bc[1] >> 16 & 0xFF) << 24);
    cd.y = (bc[2] & 0xFF) | ((bc[2] >> 16 & 0xFF) << 8) | ((bc[3] & 0xFF) << 16) | ((bc[3] >> 16 & 0xFF) << 24);
    *reinterpret_cast<uint2*>(code + o * p.o_cp + c0) = cd;
  }
}

// ---------------------------------------------------------------- image import / pyramid / plain pool ----------
// NCHW fp32 (Torch boundary) -> NHWC bf16 with C <= 8: one thread per pixel, coalesced plane reads, one 16-byte store
__global__ void __launch_bounds__(256) import_nchw_c8_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int C, int64_t HW, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int64_t n = i / HW, r = i - n * HW;
  V8 v;
#pragma unroll
  for (int c = 0; c < 8; ++c) v.v[c] = c < C ? src[(n * C + c) * HW + r] : 0.f;
  *reinterpret_cast<uint4*>(dst + i * 8) = pack8(v);
}

// SpatialAveragePooling(r,r,r,r) / plain SpatialMaxPooling(2,2,2,2):ceil(): one thread per (output pixel, 8 channels)
template <bool MAX>
__global__ void __launch_bounds__(256) pool_vec_kernel(const bf16* __restrict__ in, int H, int W, int cp, int C, int r, bf16* __restrict__ out,
                                                       int Ho, int Wo, int o_cp, int c_off, int N) {
  const int V = cp >> 3;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)N * Ho * Wo * V) return;
  int n, oy, ox, vc;
  split4(i, Ho, Wo, V, n, oy, ox, vc);
  const int c0 = vc * 8;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = MAX ? -INFINITY : 0.f;
  for (int dy = 0; dy < r; ++dy)
    for (int dx = 0; dx < r; ++dx) {
      const int y = oy * r + dy, x = ox * r + dx;
      if (y >= H || x >= W) continue;
      const V8 v = ld8(in + (((int64_t)n * H + y) * W + x) * cp + c0);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (MAX) { if (v.v[e] > acc[e] || v.v[e] != v.v[e]) acc[e] = v.v[e]; }
        else acc[e] += v.v[e];
      }
    }
  V8 o;
#pragma unroll
  for (int e = 0; e < 8; ++e) o.v[e] = (c0 + e < C) ? (MAX ? acc[e] : acc[e] / (float)(r * r)) : 0.f;
  *reinterpret_cast<uint4*>(out + (((int64_t)n * Ho + oy) * Wo + ox) * o_cp + c_off + c0) = pack8(o);
}

// im2col of a k x k / stride s / pad p window over a narrow-channel image (the ImageNet stem: 7x7, stride 2, 3 channels):
// col[n][oy][ox][ci*k*k + ky*k + kx] = in[n][oy*s - p + ky][ox*s - p + kx][ci] (0 outside), channel order = Torch's weight
// layout [Cout][Cin][k][k] flattened, so the convolution becomes a 1x1 convolution over `col` with the SAME weight
// and gradWeight storage.  One thread = 8 consecutive col channels (one 16-byte store); the 2-byte gathers hit L1.
__global__ void __launch_bounds__(256) im2col_bf16_kernel(const bf16* __restrict__ in, int H, int W, int cp_in, int C, int k, int stride, int pad,
                                                          bf16* __restrict__ col, int Ho, int Wo, int cp_col, int N) {
  pdl_launch();
  pdl_wait();
  const int V = cp_col >> 3;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)N * Ho * Wo * V) return;
  int n, oy, ox, vc;
  split4(i, Ho, Wo, V, n, oy, ox, vc);
  const int kk = k * k, K = C * kk;
  const bf16* img = in + (int64_t)n * H * W * cp_in;
  const unsigned short* img16 = reinterpret_cast<const unsigned short*>(img);
  uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = vc * 8 + e;
    unsigned short v = 0;
    if (c < K) {
      const int ci = c / kk, tap = c - ci * kk;
      const int ky = tap / k, kx = tap - ky * k;
      const int y = oy * stride - pad + ky, x = ox * stride - pad + kx;
      if ((unsigned)y < (unsigned)H && (unsigned)x < (unsigned)W) v = __ldg(img16 + ((int64_t)y * W + x) * cp_in + ci);
    }
    w[e >> 1] |= (uint32_t)v << (16 * (e & 1));
  }
  *reinterpret_cast<uint4*>(col + i * 8) = make_uint4(w[0], w[1], w[2], w[3]);
}

// ---------------------------------------------------------------- dropout ----------
// nn.Dropout in training mode (mgconv.h: mg_dropout).  One thread per (pixel, 8 channels of the pitch), one 16-byte store.  A
// vector whose 8 channels lie in one segment, starting at a multiple of 8 of its channels, is read with one 16-byte load; any
// other (segments whose C is not a multiple of 8) element by element.  Same expressions as dropout_fwd_kernel (elementwise.cu).
__global__ void __launch_bounds__(256) dropout_fwd_bf16_kernel(const __grid_constant__ DropSegs<bf16> d, const DropK k, bf16* __restrict__ out,
                                                               int N, int H, int W, int C, int V) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)N * H * W * V) return;
  int n, y, x, vc;
  split4(i, H, W, V, n, y, x, vc);
  const int64_t pix = ((int64_t)n * H + y) * W + x;
  const int c0 = vc * 8, nl = min(8, C - c0);
  V8 o;
#pragma unroll
  for (int e = 0; e < 8; ++e) o.v[e] = 0.f;
  if (nl > 0) {
    const uint32_t keep = drop_keep_bits((uint64_t)pix * C + c0, nl, k);
    int s = 0;
    while (s + 1 < d.n && c0 >= d.off[s + 1]) ++s;
    const GridV<bf16>& G = d.g[s];
    const int lc = c0 - d.off[s];
    if (nl == 8 && c0 + 8 <= d.off[s + 1] && lc % 8 == 0 && !G.scale) {
      const int yy = d.up[s] ? y >> 1 : y, xx = d.up[s] ? x >> 1 : x;
      const V8 v = ld8(G.data + (((int64_t)n * G.H + yy) * G.W + xx) * G.Cp + lc);
#pragma unroll
      for (int e = 0; e < 8; ++e) o.v[e] = (keep >> e & 1u) ? v.v[e] * k.s : 0.f;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (e < nl && (keep >> e & 1u)) o.v[e] = drop_gather(d, n, y, x, c0 + e) * k.s;
    }
  }
  *reinterpret_cast<uint4*>(out + i * 8) = pack8(o);
}

// in place g = g * mask * s, 8 channels (one 16-byte load and store) per thread; pad channels are stored back unchanged
__global__ void __launch_bounds__(256) dropout_bwd_bf16_kernel(const DropK k, bf16* __restrict__ g, int64_t P, int C, int V) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P * V) return;
  int64_t pix; int vc;
  if (i < ((int64_t)1 << 32)) { const uint32_t q = (uint32_t)i / (uint32_t)V; pix = q; vc = (int)((uint32_t)i - q * (uint32_t)V); }
  else { pix = i / V; vc = (int)(i - pix * V); }
  const int c0 = vc * 8, nl = min(8, C - c0);
  if (nl <= 0) return;
  const uint32_t keep = drop_keep_bits((uint64_t)pix * C + c0, nl, k);
  V8 v = ld8(g + i * 8);
#pragma unroll
  for (int e = 0; e < 8; ++e)
    if (e < nl) v.v[e] = (keep >> e & 1u) ? v.v[e] * k.s : 0.f;
  *reinterpret_cast<uint4*>(g + i * 8) = pack8(v);
}

static inline unsigned grid_for(int64_t threads) { return (unsigned)mg_cdiv(threads, 256); }
// persistent-style grid for the reducing kernels: a few CTAs per SM, each thread loops
static inline unsigned reduce_grid(const mg_ctx* ctx, int64_t items, int per_sm = 4) {
  // every CTA ends with 2*C global atomics: keep the grid at a few resident CTAs per SM and let threads loop
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(mg_cdiv(items, 256), (int64_t)ctx->num_sms * per_sm));
}

}  // namespace

// ---- entry points used by elementwise.cu; return false when the fast path does not apply -------------
bool bf16_apply(mg_ctx* ctx, const mg_grid* z, const mg_grid* s, int relu, mg_grid* out, mg_grid* pooled, const mg_bn_fused* bn) {
  if (s && (s->scale || s->Cp % 8)) return false;
  if (z->Cp % 8 || out->Cp % 8 || z->Cp < out->Cp) return false;
  if (pooled && pooled->Cp % 8) return false;
  if (bn && (!z->scale || !z->shift || z->Cp > 4096)) return false;
  ApplyP p;
  memset(&p, 0, sizeof(p));
  if (bn) {
    p.bn = 1; p.training = bn->training; p.sums = bn->sums; p.count = bn->count; p.gamma = bn->gamma; p.beta = bn->beta;
    p.rmean = bn->running_mean; p.rvar = bn->running_var; p.eps = bn->eps; p.momentum = bn->momentum;
    p.smean = bn->save_mean; p.sinvstd = bn->save_invstd; p.scale_out = const_cast<float*>(z->scale); p.shift_out = const_cast<float*>(z->shift);
    p.inv_count = 1.0 / (double)bn->count; p.unbias = bn->count > 1 ? (double)bn->count / (double)(bn->count - 1) : 1.0;
  }
  p.z = (const bf16*)z->data; p.z_cp = z->Cp; p.scale = z->scale; p.shift = z->shift; p.z_relu = z->relu;
  p.s = s ? (const bf16*)s->data : nullptr; p.s_cp = s ? s->Cp : 0;
  p.relu = relu; p.out = (bf16*)out->data; p.o_cp = out->Cp;
  p.pooled = pooled ? (bf16*)pooled->data : nullptr; p.p_cp = pooled ? pooled->Cp : 0;
  p.N = z->N; p.H = z->H; p.W = z->W; p.C = z->C; p.Hp = (z->H + 1) / 2; p.Wp = (z->W + 1) / 2;
  if (out->Cp > 2048) return false;
  const int64_t total = (int64_t)p.N * p.Hp * p.Wp * (p.o_cp / 8);
  if (total >= ((int64_t)1 << 31) || (int64_t)p.N * p.H * p.W >= ((int64_t)1 << 31)) return false;   // 32-bit index decode
  p.fd_v = make_fastdiv((uint32_t)(p.o_cp / 8)); p.fd_wp = make_fastdiv((uint32_t)p.Wp); p.fd_hp = make_fastdiv((uint32_t)p.Hp);
  // one 2x2 block x 8 channels per thread (measured: looping CTAs with batched loads need 80 registers and lose 10-40 %)
  static int per_sm = -1;
  if (per_sm < 0) { const char* e = getenv("MGCONV_APPLY_CTAS"); per_sm = e ? atoi(e) : 6; }
  const unsigned grid = (unsigned)std::min<int64_t>(grid_for(total), (int64_t)per_sm * ctx->num_sms);
  mg_launch_pdl(apply_bf16_kernel, dim3(grid), dim3(256), bn ? 2 * z->Cp * sizeof(float) : 0, ctx->stream, p);
  return true;
}

bool bf16_bn_stats(mg_ctx* ctx, const mg_grid* y, mg_sum* sums) {
  if (y->Cp % 8 || y->Cp > 2048) return false;
  const int64_t P = (int64_t)y->N * y->H * y->W;
  const int V = y->Cp / 8;
  mg_launch_pdl(bn_stats_bf16_kernel, dim3(reduce_grid(ctx, P * V / 4)), dim3(256), 2 * 256 * 8 * sizeof(float), ctx->stream, (const bf16*)y->data, y->Cp, y->C, P, sums);
  return true;
}

bool bf16_combine(mg_ctx* ctx, const mg_grid* x, int relu_mask, const mg_grid* bn_x, int n_src, const mg_grad_src* src, mg_grid* d,
                  mg_sum* sums, const FrozenBn* fz) {
  const mg_grid* o = fz ? fz->g : d;   // the tensor the pass writes in full (G when frozen; d may then be null)
  if (x->Cp % 8 || o->Cp % 8 || o->Cp > 2048 || x->scale || x->Cp < o->Cp) return false;
  if (fz && d && d->Cp != o->Cp) return false;
  if (relu_mask == 2 && !(n_src == 1 && src[0].mode == 3 && src[0].aux && bn_x)) return false;   // x = pooled tensor of the stem's mode-3 source
  if (sums && bn_x && bn_x->Cp < o->Cp) return false;
  CombP p;
  memset(&p, 0, sizeof(p));
  for (int s = 0; s < n_src; ++s) {
    const mg_grad_src& g = src[s];
    if (g.c_offset % 8 || g.g.Cp % 8 || g.c_offset + o->Cp > g.g.Cp) return false;
    if (g.mode == 3 && !g.aux) return false;
    p.src[s].g = (const bf16*)g.g.data; p.src[s].aux = (const uint8_t*)g.aux;
    p.src[s].H = g.g.H; p.src[s].W = g.g.W; p.src[s].cp = g.g.Cp; p.src[s].c_off = g.c_offset; p.src[s].mode = g.mode;
  }
  p.n_src = n_src;
  p.x = (const bf16*)x->data; p.x_cp = x->Cp;
  const mg_grid* bx = bn_x ? bn_x : x;
  p.bnx = (const bf16*)bx->data; p.bn_cp = bx->Cp;
  p.relu_mask = relu_mask; p.d = d ? (bf16*)d->data : nullptr; p.d_cp = o->Cp; p.sums = sums;
  p.g = fz ? (bf16*)fz->g->data : nullptr; p.g_cp = o->Cp;
  if (fz) { p.fz_gamma = fz->gamma; p.fz_rvar = fz->running_var; p.fz_eps = fz->eps; }
  p.N = o->N; p.H = o->H; p.W = o->W; p.C = o->C; p.Hb = (o->H + 1) / 2; p.Wb = (o->W + 1) / 2;
  const int V = o->Cp / 8;
  const int64_t items = (int64_t)p.N * p.Hb * p.Wb * V;
  static int spec = -1;
  if (spec < 0) { const char* e = getenv("MGCONV_COMBINE_SPEC"); spec = e ? atoi(e) : 1; }
  static int fast_env = -1;   // batched-load form of the specialised kernels (MGCONV_COMBINE_FAST=0: the older form, for A/B timing)
  if (fast_env < 0) { const char* e = getenv("MGCONV_COMBINE_FAST"); fast_env = e ? atoi(e) : 1; }
  bool fast = (fast_env != 0 || relu_mask == 2) && (int64_t)p.N * p.H * p.W < ((int64_t)1 << 31);   // 32-bit pixel indices (of the finer source grids too)
  for (int s = 0; s < n_src; ++s) fast = fast && (int64_t)src[s].g.N * src[s].g.H * src[s].g.W < ((int64_t)1 << 31);
  p.fd_wb = make_fastdiv((uint32_t)p.Wb); p.fd_hb = make_fastdiv((uint32_t)p.Hb);
  int code = 0;
  for (int s = 0; s < n_src; ++s) code |= (src[s].mode & 3) << (2 * s);
  const size_t smem = sums ? 2 * 256 * 8 * sizeof(float) : 0;   // block_channel_sums staging
  // the source-mode lists of the multigrid builders (same / pool / up gathers of ResampleConcat + shortcut); anything else
  // takes the generic kernel.  Frozen BatchNorm: the specialised batched-load kernels only (false otherwise: the caller then runs
  // the generic kernel of elementwise.cu)
  if (fz && !(spec && fast)) return false;
#define MG_COMBINE_CASE(NSRC, M0, M1, M2, M3)                                                                      \
  if (spec && n_src == NSRC && code == ((M0) | (M1) << 2 | (M2) << 4 | (M3) << 6)) {                                  \
    if (fz)                                                                                                          \
      mg_launch_pdl(combine_fast_kernel<NSRC, ((M0) | (M1) << 2 | (M2) << 4 | (M3) << 6), true>, dim3(reduce_grid(ctx, items, 1)), \
                    dim3(256), 2 * 256 * 8 * sizeof(float) + o->Cp * sizeof(float), ctx->stream, p);                \
    else if (fast)                                                                                                   \
      mg_launch_pdl(combine_fast_kernel<NSRC, ((M0) | (M1) << 2 | (M2) << 4 | (M3) << 6), false>, dim3(reduce_grid(ctx, items, 2)), \
                    dim3(256), smem, ctx->stream, p);                                                                \
    else                                                                                                             \
      mg_launch_pdl(combine_bf16_kernel<NSRC, ((M0) | (M1) << 2 | (M2) << 4 | (M3) << 6)>, dim3(reduce_grid(ctx, items, 2)), \
                    dim3(256), smem, ctx->stream, p);                                                                \
    return true;                                                                                                     \
  }
  MG_COMBINE_CASE(1, 0, 0, 0, 0)
  MG_COMBINE_CASE(1, 1, 0, 0, 0)
  MG_COMBINE_CASE(1, 3, 0, 0, 0)
  MG_COMBINE_CASE(2, 0, 0, 0, 0)
  MG_COMBINE_CASE(2, 0, 1, 0, 0)
  MG_COMBINE_CASE(2, 0, 2, 0, 0)
  MG_COMBINE_CASE(2, 1, 1, 0, 0)
  MG_COMBINE_CASE(3, 0, 0, 1, 0)
  MG_COMBINE_CASE(3, 0, 0, 2, 0)
  MG_COMBINE_CASE(3, 0, 2, 1, 0)
  MG_COMBINE_CASE(4, 0, 0, 2, 1)
#undef MG_COMBINE_CASE
  if (fz) return false;
  const unsigned grid = reduce_grid(ctx, items, 3);   // 80 registers: three CTAs per SM are resident
  mg_launch_pdl(combine_bf16_kernel<-1, 0>, dim3(grid), dim3(256), smem, ctx->stream, p);
  return true;
}

bool bf16_bn_bwd_apply(mg_ctx* ctx, const mg_grid* xraw, const mg_grid* d, mg_grid* out, const mg_sum* sums, int64_t count, const float* gamma,
                       const float* mean, const float* invstd, float* dgamma, float* dbeta, float* conv_dbias, float gscale) {
  if (xraw->Cp % 8 || d->Cp % 8 || out->Cp % 8 || d->Cp != out->Cp || xraw->Cp < out->Cp || out->Cp > 2048) return false;
  BnBwdP bp;
  bp.sums = sums; bp.count = count; bp.inv_count = 1.0 / (double)count; bp.gamma = gamma; bp.mean = mean; bp.invstd = invstd; bp.dgamma = dgamma; bp.dbeta = dbeta;
  const int64_t P = (int64_t)d->N * d->H * d->W;
  const int V = out->Cp / 8;
  const unsigned grid = reduce_grid(ctx, P * V, 4);
  mg_launch_pdl(bn_bwd_apply_bf16_kernel, dim3(grid), dim3(256), 3 * V * 8 * sizeof(float), ctx->stream, (const bf16*)xraw->data, xraw->Cp,
                (const bf16*)d->data, d->Cp, (bf16*)out->data, out->Cp, d->C, P, bp, conv_dbias, gscale);
  return true;
}

bool bf16_pool3(mg_ctx* ctx, const mg_grid* in, mg_grid* out, uint8_t* code) {
  if (in->Cp % 8 || in->Cp != out->Cp || in->scale) return false;
  const int64_t total = (int64_t)in->N * out->H * out->W * (in->Cp / 8);
  pool3_bf16_kernel<<<grid_for(total), 256, 0, ctx->stream>>>((const bf16*)in->data, in->H, in->W, in->Cp, in->C, (bf16*)out->data, code,
                                                             out->H, out->W, in->N);
  return true;
}

bool bf16_bn_relu_pool3(mg_ctx* ctx, const mg_grid* z, const mg_bn_fused* bn, mg_grid* out, uint8_t* code) {
  if (z->Cp % 8 || out->Cp != z->Cp || z->Cp > 4096 || !z->scale || !z->shift || !code) return false;
  const int64_t total = (int64_t)z->N * out->H * out->W * (z->Cp / 8);
  if (total >= ((int64_t)1 << 31) || (int64_t)z->N * z->H * z->W >= ((int64_t)1 << 31)) return false;
  ApplyP p;
  memset(&p, 0, sizeof(p));
  p.bn = 1; p.training = bn->training; p.sums = bn->sums; p.count = bn->count; p.gamma = bn->gamma; p.beta = bn->beta;
  p.rmean = bn->running_mean; p.rvar = bn->running_var; p.eps = bn->eps; p.momentum = bn->momentum;
  p.smean = bn->save_mean; p.sinvstd = bn->save_invstd; p.scale_out = const_cast<float*>(z->scale); p.shift_out = const_cast<float*>(z->shift);
  p.inv_count = 1.0 / (double)bn->count; p.unbias = bn->count > 1 ? (double)bn->count / (double)(bn->count - 1) : 1.0;
  p.z = (const bf16*)z->data; p.z_cp = z->Cp; p.out = (bf16*)out->data; p.o_cp = out->Cp;
  p.N = z->N; p.H = z->H; p.W = z->W; p.C = z->C;
  p.fd_v = make_fastdiv((uint32_t)(p.o_cp / 8)); p.fd_wp = make_fastdiv((uint32_t)out->W); p.fd_hp = make_fastdiv((uint32_t)out->H);
  const unsigned grid = (unsigned)std::min<int64_t>(grid_for(total), (int64_t)6 * ctx->num_sms);
  mg_launch_pdl(bn_relu_pool3_bf16_kernel, dim3(grid), dim3(256), 2 * z->Cp * sizeof(float), ctx->stream, p, code, out->H, out->W);
  return true;
}

bool bf16_import_nchw(mg_ctx* ctx, const float* src, mg_grid* dst) {
  if (dst->Cp != 8) return false;
  const int64_t HW = (int64_t)dst->H * dst->W, total = HW * dst->N;
  import_nchw_c8_kernel<<<grid_for(total), 256, 0, ctx->stream>>>(src, (bf16*)dst->data, dst->C, HW, total);
  return true;
}

bool bf16_im2col(mg_ctx* ctx, const mg_grid* in, int k, int stride, int pad, mg_grid* col) {
  if (in->scale || col->Cp % 8) return false;
  const int64_t total = (int64_t)in->N * col->H * col->W * (col->Cp / 8);
  mg_launch_pdl(im2col_bf16_kernel, dim3(grid_for(total)), dim3(256), 0, ctx->stream, (const bf16*)in->data, in->H, in->W, in->Cp, in->C, k, stride,
                pad, (bf16*)col->data, col->H, col->W, col->Cp, in->N);
  return true;
}

bool bf16_avgpool(mg_ctx* ctx, const mg_grid* in, int r, mg_grid* out) {
  if (in->scale || in->Cp % 8 || out->Cp != in->Cp) return false;
  const int64_t total = (int64_t)in->N * out->H * out->W * (in->Cp / 8);
  pool_vec_kernel<false><<<grid_for(total), 256, 0, ctx->stream>>>((const bf16*)in->data, in->H, in->W, in->Cp, in->C, r, (bf16*)out->data,
                                                                   out->H, out->W, out->Cp, 0, in->N);
  return true;
}

bool bf16_dropout_forward(mg_ctx* ctx, const DropK& k, int n_seg, const mg_grid* seg, const int32_t* mode, mg_grid* out) {
  for (int s = 0; s < n_seg; ++s)
    if (seg[s].Cp % 8) return false;
  const int V = out->Cp / 8;
  const int64_t total = (int64_t)out->N * out->H * out->W * V;
  dropout_fwd_bf16_kernel<<<grid_for(total), 256, 0, ctx->stream>>>(make_drop_segs<bf16>(n_seg, seg, mode), k, (bf16*)out->data, out->N, out->H,
                                                                    out->W, out->C, V);
  return true;
}

bool bf16_dropout_backward(mg_ctx* ctx, const DropK& k, mg_grid* g) {
  const int V = g->Cp / 8;
  const int64_t P = (int64_t)g->N * g->H * g->W;
  dropout_bwd_bf16_kernel<<<grid_for(P * V), 256, 0, ctx->stream>>>(k, (bf16*)g->data, P, g->C, V);
  return true;
}

bool bf16_pool2(mg_ctx* ctx, const mg_grid* in, mg_grid* out, int c_off) {
  if (in->scale || in->Cp % 8 || out->Cp % 8 || c_off % 8 || c_off + in->Cp > out->Cp) return false;
  const int64_t total = (int64_t)in->N * out->H * out->W * (in->Cp / 8);
  pool_vec_kernel<true><<<grid_for(total), 256, 0, ctx->stream>>>((const bf16*)in->data, in->H, in->W, in->Cp, in->C, 2, (bf16*)out->data,
                                                                  out->H, out->W, out->Cp, c_off, in->N);
  return true;
}
