// Plan-level C ABI: one multigrid STAGE -- the residual mg-unit of models/ilsvrc/rnmg.lua:91-159 (or the plain mgConv of
// models/cifar/nmg.lua:31-86) -- as a single pair of entry points that take and return what the reference's modules take and
// return: one NCHW fp32 device tensor per grid, finest first, plus the Torch-layout parameters.  Everything the Python host does
// per stage in lower.py / ops.py (segment lists, pooled companions, epilogue fusion, gradient routing in gather form) is done
// here in C++, so a Lua host needs nothing but `ffi.cdef` of mgconv.h: lua/mgconv_nn.lua is a thin nn.Module around these calls.
//
//   x_i --import--> X_i (NHWC bf16/fp32) --maxpool2x2 ceil--> P(X_i)                                      rnmg.lua:53-60
//   layer 1, grid i:  y1_i = conv(cat[P(X_{i-1}) | X_i | up(X_{i+1})]),  a1_i = relu(BN(y1_i)) (+ P(a1_i))    rnmg.lua:104-117
//   layer 2, grid i:  y2_i = conv(cat[P(a1_{i-1}) | a1_i | up(a1_{i+1})]), out_i = relu(BN(y2_i) + pad(X_i))   rnmg.lua:118-154
//   backward: gradients are combined per tensor in gather form (mg_grad_combine), BN backward, wgrad, dgrad.
#include "common.cuh"
#include <new>

struct mg_stage_plan {
  mg_ctx* ctx;
  mg_stage_desc d;
  int batch, n, layers, elt;
  int last_training;   // training flag of the last mg_stage_forward (-1: none yet); mg_stage_backward differentiates that mode
  int grad_input_ready;   // mg_stage_update_grad_input ran since the last mg_stage_forward: mg_stage_acc_grad_parameters may follow
  // byte offsets into the workspace
  size_t X[MG_STAGE_MAX_GRIDS], PX[MG_STAGE_MAX_GRIDS], DX[MG_STAGE_MAX_GRIDS], DY[MG_STAGE_MAX_GRIDS];
  size_t y[2][MG_STAGE_MAX_GRIDS], a[2][MG_STAGE_MAX_GRIDS], Pa[2][MG_STAGE_MAX_GRIDS];
  size_t D[2][MG_STAGE_MAX_GRIDS], G[2][MG_STAGE_MAX_GRIDS], dcat[2][MG_STAGE_MAX_GRIDS];
  size_t wpack[2][MG_STAGE_MAX_GRIDS], wpack_t[2][MG_STAGE_MAX_GRIDS];
  size_t fsums[2][MG_STAGE_MAX_GRIDS], bsums[2][MG_STAGE_MAX_GRIDS];
  size_t scale[2][MG_STAGE_MAX_GRIDS], shift[2][MG_STAGE_MAX_GRIDS], mean[2][MG_STAGE_MAX_GRIDS], invstd[2][MG_STAGE_MAX_GRIDS], coef[2][MG_STAGE_MAX_GRIDS];
  size_t sums_begin, sums_bytes;      // all forward + backward sums are contiguous: one memset per pass
  size_t bytes;
  int ccatp[2][MG_STAGE_MAX_GRIDS];   // padded width of the concatenated input of conv (layer, grid)
};

namespace {

inline int cpad(int c) { return (c + 7) / 8 * 8; }
inline size_t al(size_t b) { return (b + 255) & ~(size_t)255; }

inline mg_grid grid_of(void* ws, size_t off, int N, int H, int W, int C, const float* scale = nullptr, const float* shift = nullptr) {
  mg_grid g;
  g.data = (char*)ws + off; g.scale = scale; g.shift = shift; g.relu = 0;
  g.N = N; g.H = H; g.W = W; g.C = C; g.Cp = cpad(C);
  return g;
}

// channels of the tensors that enter layer `l` (0: the unit's inputs, 1: the first layer's outputs)
inline int cin_of(const mg_stage_desc& d, int l, int i) { return l == 0 ? d.C_in[i] : d.C_out[i]; }

// conv descriptor of (layer l, grid i) over the workspace `ws`
void make_desc(const mg_stage_plan* p, void* ws, int l, int i, mg_conv_desc* cd) {
  const mg_stage_desc& d = p->d;
  memset(cd, 0, sizeof(*cd));
  int s = 0;
  const size_t* src = l == 0 ? p->X : p->a[0];
  const size_t* psrc = l == 0 ? p->PX : p->Pa[0];
  if (i > 0) {            // finer grid through its pooled companion (SpatialMaxPooling(2,2,2,2):ceil())
    cd->seg[s] = grid_of(ws, psrc[i - 1], p->batch, d.H[i], d.W[i], cin_of(d, l, i - 1));
    cd->seg_mode[s++] = MG_SEG_SAME;
  }
  cd->seg[s] = grid_of(ws, src[i], p->batch, d.H[i], d.W[i], cin_of(d, l, i));
  cd->seg_mode[s++] = MG_SEG_SAME;
  if (i + 1 < p->n) {     // coarser grid, up-sampled by the conv's loader (SpatialUpSamplingNearest(2))
    cd->seg[s] = grid_of(ws, src[i + 1], p->batch, d.H[i + 1], d.W[i + 1], cin_of(d, l, i + 1));
    cd->seg_mode[s++] = MG_SEG_UP;
  }
  cd->n_seg = s;
  cd->ksize = d.ksize[i]; cd->stride = 1; cd->pad = d.ksize[i] / 2; cd->Cout = d.C_out[i];
  cd->H = d.H[i]; cd->W = d.W[i];
}

}  // namespace

extern "C" {

int mg_plan_create(mg_ctx* ctx, const mg_stage_desc* d, int32_t batch, mg_stage_plan** out) {
  if (!ctx || !d || !out || batch < 1) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, d->n_scales >= 1 && d->n_scales <= MG_STAGE_MAX_GRIDS, MG_ERR_INVALID_ARG, "plan: %d grids (1..%d)", d->n_scales, MG_STAGE_MAX_GRIDS);
  for (int i = 0; i < d->n_scales; ++i) {
    MG_REQUIRE(ctx, d->C_in[i] >= 1 && d->C_out[i] >= 1 && d->H[i] >= 1 && d->W[i] >= 1, MG_ERR_INVALID_ARG, "plan: grid %d has an empty dimension", i);
    MG_REQUIRE(ctx, d->ksize[i] == 1 || d->ksize[i] == 3, MG_ERR_UNSUPPORTED, "plan: kernel size %d on grid %d (1 or 3)", d->ksize[i], i);
    MG_REQUIRE(ctx, !d->residual || d->C_in[i] <= d->C_out[i], MG_ERR_UNSUPPORTED,
               "plan: the shortcut of grid %d would need a projection (%d -> %d channels); nn.Padding only appends", i, d->C_in[i], d->C_out[i]);
    if (i + 1 < d->n_scales)   // JoinTable(2) of ResampleConcat raises the same size error in the reference
      MG_REQUIRE(ctx, d->H[i] == 2 * d->H[i + 1] && d->W[i] == 2 * d->W[i + 1], MG_ERR_SHAPE, "plan: grid %d is %dx%d, grid %d is %dx%d (must halve)",
                 i, d->H[i], d->W[i], i + 1, d->H[i + 1], d->W[i + 1]);
  }
  mg_stage_plan* p = new (std::nothrow) mg_stage_plan();
  MG_REQUIRE(ctx, p != nullptr, MG_ERR_INVALID_ARG, "plan: out of memory");
  memset(p, 0, sizeof(*p));
  p->ctx = ctx; p->d = *d; p->batch = batch; p->n = d->n_scales; p->layers = d->residual ? 2 : 1;
  p->elt = (int)mg_elt_size(ctx->dtype);
  p->last_training = -1;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += al(bytes); return o; };
  const int n = p->n, L = p->layers;
  for (int i = 0; i < n; ++i) {
    const size_t px = (size_t)batch * d->H[i] * d->W[i];
    p->X[i] = take(px * cpad(d->C_in[i]) * p->elt);
    p->DX[i] = take(px * cpad(d->C_in[i]) * p->elt);
    p->DY[i] = take(px * cpad(d->C_out[i]) * p->elt);
    if (i + 1 < n) p->PX[i] = take((size_t)batch * d->H[i + 1] * d->W[i + 1] * cpad(d->C_in[i]) * p->elt);
    for (int l = 0; l < L; ++l) {
      p->y[l][i] = take(px * cpad(d->C_out[i]) * p->elt);
      p->a[l][i] = take(px * cpad(d->C_out[i]) * p->elt);
      if (i + 1 < n && l + 1 < L) p->Pa[l][i] = take((size_t)batch * d->H[i + 1] * d->W[i + 1] * cpad(d->C_out[i]) * p->elt);
      p->D[l][i] = take(px * cpad(d->C_out[i]) * p->elt);
      p->G[l][i] = take(px * cpad(d->C_out[i]) * p->elt);
      int cc = cpad(cin_of(*d, l, i));
      if (i > 0) cc += cpad(cin_of(*d, l, i - 1));
      if (i + 1 < n) cc += cpad(cin_of(*d, l, i + 1));
      p->ccatp[l][i] = cc;
      p->dcat[l][i] = take(px * cc * p->elt);
      const size_t cp4 = (size_t)cpad(d->C_out[i]) * sizeof(float);
      p->scale[l][i] = take(cp4); p->shift[l][i] = take(cp4); p->mean[l][i] = take(cp4); p->invstd[l][i] = take(cp4); p->coef[l][i] = take(3 * cp4);
    }
  }
  // packed operand images of the tensor-core path (sizes depend on the descriptors; pointers are irrelevant for the size)
  for (int l = 0; l < L; ++l)
    for (int i = 0; i < n; ++i) {
      mg_conv_desc cd;
      make_desc(p, (void*)16, l, i, &cd);
      const size_t nb = ctx->dtype == MG_BF16 && ctx->impl != MG_IMPL_SIMT ? mg_conv_packed_bytes(&cd, 0) : 0;
      const size_t nt = ctx->dtype == MG_BF16 && ctx->impl != MG_IMPL_SIMT ? mg_conv_packed_bytes(&cd, 1) : 0;
      p->wpack[l][i] = nb ? take(nb) : (size_t)-1;
      p->wpack_t[l][i] = nt ? take(nt) : (size_t)-1;
    }
  p->sums_begin = off;
  for (int l = 0; l < L; ++l)
    for (int i = 0; i < n; ++i) {
      p->fsums[l][i] = take(2 * (size_t)d->C_out[i] * sizeof(mg_sum));
      p->bsums[l][i] = take(2 * (size_t)d->C_out[i] * sizeof(mg_sum));
    }
  p->sums_bytes = off - p->sums_begin;
  p->bytes = off;
  *out = p;
  return MG_OK;
}

size_t mg_plan_workspace_bytes(const mg_stage_plan* p) { return p ? p->bytes : 0; }

int mg_plan_destroy(mg_stage_plan* p) {
  if (!p) return MG_ERR_INVALID_ARG;
  delete p;
  return MG_OK;
}

#define MG_TRY(expr) do { int _rc = (expr); if (_rc) return _rc; } while (0)

int mg_stage_forward(mg_stage_plan* p, void* workspace, const float* const* x, const mg_stage_params* prm, float* const* y, int training) {
  if (!p || !workspace || !x || !prm || !y) return MG_ERR_INVALID_ARG;
  mg_ctx* ctx = p->ctx;
  const mg_stage_desc& d = p->d;
  const int n = p->n, L = p->layers, B = p->batch;
  char* ws = (char*)workspace;
  MG_REQUIRE(ctx, ((uintptr_t)workspace & 255) == 0, MG_ERR_INVALID_ARG, "stage_forward: workspace must be 256-byte aligned");
  MG_TRY(mg_memset_zero(ctx, ws + p->sums_begin, p->sums_bytes));
  p->last_training = training ? 1 : 0;
  p->grad_input_ready = 0;
  // inputs: NCHW fp32 -> grids, plus the pooled companion every coarser neighbour gathers
  for (int i = 0; i < n; ++i) {
    MG_REQUIRE(ctx, x[i] != nullptr, MG_ERR_INVALID_ARG, "stage_forward: x[%d] is null", i);
    mg_grid X = grid_of(ws, p->X[i], B, d.H[i], d.W[i], d.C_in[i]);
    MG_TRY(mg_import_nchw(ctx, x[i], &X));
    if (i + 1 < n) {
      mg_grid P = grid_of(ws, p->PX[i], B, d.H[i + 1], d.W[i + 1], d.C_in[i]);
      MG_TRY(mg_pool_forward(ctx, &X, &P, 0, nullptr));
    }
  }
  for (int l = 0; l < L; ++l) {
    const bool last = l + 1 == L;
    for (int i = 0; i < n; ++i) {
      const int k = l * n + i;
      MG_REQUIRE(ctx, prm->conv_w[k] && prm->conv_b[k] && prm->bn_g[k] && prm->bn_b[k] && prm->bn_rm[k] && prm->bn_rv[k], MG_ERR_INVALID_ARG,
                 "stage_forward: parameters of conv / BN %d (layer %d, grid %d) are null", k, l, i);
      mg_conv_desc cd;
      make_desc(p, ws, l, i, &cd);
      void* wp = p->wpack[l][i] == (size_t)-1 ? nullptr : ws + p->wpack[l][i];
      if (wp) MG_TRY(mg_conv_pack_weights(ctx, &cd, prm->conv_w[k], wp, 0));
      mg_grid Y = grid_of(ws, p->y[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      mg_sum* sums = (mg_sum*)(ws + p->fsums[l][i]);
      // evaluation mode normalises with the running statistics: the epilogue reduces no batch statistics
      MG_TRY(mg_conv_forward(ctx, &cd, prm->conv_w[k], wp, prm->conv_b[k], &Y, training ? sums : nullptr));
      // SpatialBatchNormalization -> [CAddTable with the (padded) shortcut] -> [ReLU] -> [pooled companion], one pass
      mg_grid Z = grid_of(ws, p->y[l][i], B, d.H[i], d.W[i], d.C_out[i], (const float*)(ws + p->scale[l][i]), (const float*)(ws + p->shift[l][i]));
      mg_bn_fused f;
      memset(&f, 0, sizeof(f));
      f.sums = sums; f.count = (int64_t)B * d.H[i] * d.W[i];
      f.gamma = prm->bn_g[k]; f.beta = prm->bn_b[k]; f.running_mean = prm->bn_rm[k]; f.running_var = prm->bn_rv[k];
      f.eps = d.eps; f.momentum = d.momentum; f.training = training ? 1 : 0;
      f.save_mean = (float*)(ws + p->mean[l][i]); f.save_invstd = (float*)(ws + p->invstd[l][i]);
      mg_grid A = grid_of(ws, p->a[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      mg_grid S = grid_of(ws, p->X[i], B, d.H[i], d.W[i], d.C_in[i]);
      mg_grid PA;
      const bool want_pool = !last && i + 1 < n;
      if (want_pool) PA = grid_of(ws, p->Pa[l][i], B, d.H[i + 1], d.W[i + 1], d.C_out[i]);
      const int relu = last ? (d.no_final_relu ? 0 : 1) : 1;
      MG_TRY(mg_bn_residual_forward(ctx, &Z, &f, (last && d.residual) ? &S : nullptr, relu, &A, want_pool ? &PA : nullptr));
      if (last) {
        MG_REQUIRE(ctx, y[i] != nullptr, MG_ERR_INVALID_ARG, "stage_forward: y[%d] is null", i);
        MG_TRY(mg_export_nchw(ctx, &A, y[i]));
      }
    }
  }
  return MG_OK;
}

}  // extern "C"

namespace {

// mg_stage_backward (params: every gradient) and mg_stage_update_grad_input (!params: the data gradient alone -- BatchNorm
// with dgamma / dbeta / conv_dbias NULL, no weight gradient; the sums of every layer stay in the workspace for
// mg_stage_acc_grad_parameters)
int stage_backward(mg_stage_plan* p, void* workspace, const float* const* dy, const mg_stage_params* prm, float* const* dx, float scale,
                   bool params, const char* who) {
  if (!p || !workspace || !dy || !prm) return MG_ERR_INVALID_ARG;
  mg_ctx* ctx = p->ctx;
  const mg_stage_desc& d = p->d;
  const int n = p->n, L = p->layers, B = p->batch;
  char* ws = (char*)workspace;
  MG_REQUIRE(ctx, p->last_training >= 0, MG_ERR_INVALID_ARG, "%s: no mg_stage_forward on this plan yet", who);
  const bool frozen = p->last_training == 0;
  for (int i = 0; i < n; ++i) {
    MG_REQUIRE(ctx, dy[i] != nullptr, MG_ERR_INVALID_ARG, "stage_backward: dy[%d] is null", i);
    mg_grid DY = grid_of(ws, p->DY[i], B, d.H[i], d.W[i], d.C_out[i]);
    MG_TRY(mg_import_nchw(ctx, dy[i], &DY));
  }
  for (int l = L - 1; l >= 0; --l) {
    const bool last = l + 1 == L;
    for (int i = 0; i < n; ++i) {
      const int k = l * n + i;
      if (params)
        MG_REQUIRE(ctx, prm->conv_gw[k] && prm->conv_gb[k] && prm->bn_gg[k] && prm->bn_gb[k], MG_ERR_INVALID_ARG,
                   "%s: gradient tensors of conv / BN %d are null", who, k);
      float* const bn_gg = params ? prm->bn_gg[k] : nullptr;
      float* const bn_gb = params ? prm->bn_gb[k] : nullptr;
      float* const conv_gb = params ? prm->conv_gb[k] : nullptr;
      // gradient of a_l,i in gather form: its consumers' contributions, times its ReLU mask, plus the BN sums
      mg_grad_src src[3];
      int ns = 0;
      memset(src, 0, sizeof(src));
      if (last) {
        src[ns].g = grid_of(ws, p->DY[i], B, d.H[i], d.W[i], d.C_out[i]); src[ns].c_offset = 0; src[ns].mode = MG_SEG_SAME; ++ns;
      } else {   // consumers are the three convs of layer l+1 that gathered a_l,i: same grid, coarser (pooled), finer (up-sampled)
        const int l2 = l + 1;
        int off_same = i > 0 ? cpad(d.C_out[i - 1]) : 0;
        src[ns].g = grid_of(ws, p->dcat[l2][i], B, d.H[i], d.W[i], p->ccatp[l2][i]); src[ns].g.Cp = p->ccatp[l2][i];
        src[ns].c_offset = off_same; src[ns].mode = MG_SEG_SAME; ++ns;
        if (i + 1 < n) {   // conv (l2, i+1) read P(a_l,i) as its FIRST segment
          src[ns].g = grid_of(ws, p->dcat[l2][i + 1], B, d.H[i + 1], d.W[i + 1], p->ccatp[l2][i + 1]); src[ns].g.Cp = p->ccatp[l2][i + 1];
          src[ns].c_offset = 0; src[ns].mode = MG_SEG_POOL; ++ns;
        }
        if (i > 0) {       // conv (l2, i-1) read up(a_l,i) as its LAST segment
          const int off_up = (i - 1 > 0 ? cpad(d.C_out[i - 2]) : 0) + cpad(d.C_out[i - 1]);
          src[ns].g = grid_of(ws, p->dcat[l2][i - 1], B, d.H[i - 1], d.W[i - 1], p->ccatp[l2][i - 1]); src[ns].g.Cp = p->ccatp[l2][i - 1];
          src[ns].c_offset = off_up; src[ns].mode = MG_SEG_UP; ++ns;
        }
      }
      mg_grid A = grid_of(ws, p->a[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      mg_grid Yraw = grid_of(ws, p->y[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      mg_grid Dg = grid_of(ws, p->D[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      mg_grid Gg = grid_of(ws, p->G[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      mg_sum* bs = (mg_sum*)(ws + p->bsums[l][i]);
      MG_TRY(mg_memset_zero(ctx, bs, 2 * (size_t)d.C_out[i] * sizeof(mg_sum)));
      const int relu = last ? (d.no_final_relu ? 0 : 1) : 1;
      if (frozen) {   // evaluation-mode BatchNorm: G = gamma * invstd_r * D in the combine pass; D itself only for the shortcut
        MG_TRY(mg_grad_combine_bn_frozen(ctx, &A, relu, &Yraw, ns, src, prm->bn_g[k], prm->bn_rv[k], d.eps, &Gg, (last && d.residual) ? &Dg : nullptr, bs));
        if (params)
          MG_TRY(mg_bn_backward_frozen(ctx, bs, d.C_out[i], prm->bn_g[k], prm->bn_rm[k], prm->bn_rv[k], d.eps, bn_gg, bn_gb, scale, conv_gb));
      } else {
        MG_TRY(mg_grad_combine(ctx, &A, relu, &Yraw, ns, src, &Dg, bs));
        MG_TRY(mg_bn_backward(ctx, &Yraw, &Dg, &Gg, bs, (int64_t)B * d.H[i] * d.W[i], prm->bn_g[k], (const float*)(ws + p->mean[l][i]),
                              (const float*)(ws + p->invstd[l][i]), bn_gg, bn_gb, scale, (float*)(ws + p->coef[l][i]), conv_gb));
      }
      mg_conv_desc cd;
      make_desc(p, ws, l, i, &cd);
      if (params) MG_TRY(mg_conv_backward_weight(ctx, &cd, &Gg, prm->conv_gw[k], nullptr, scale));
      void* wpt = p->wpack_t[l][i] == (size_t)-1 ? nullptr : ws + p->wpack_t[l][i];
      if (wpt) MG_TRY(mg_conv_pack_weights(ctx, &cd, prm->conv_w[k], wpt, 1));
      mg_grid DC = grid_of(ws, p->dcat[l][i], B, d.H[i], d.W[i], p->ccatp[l][i]);
      DC.Cp = p->ccatp[l][i];
      MG_TRY(mg_conv_backward_data(ctx, &cd, prm->conv_w[k], wpt, &Gg, &DC));
    }
  }
  if (!dx) return MG_OK;
  // gradient of the unit's inputs: the three convs of layer 0 that gathered X_i, plus the shortcut
  for (int i = 0; i < n; ++i) {
    if (!dx[i]) continue;
    mg_grad_src src[4];
    int ns = 0;
    memset(src, 0, sizeof(src));
    const int off_same = i > 0 ? cpad(d.C_in[i - 1]) : 0;
    src[ns].g = grid_of(ws, p->dcat[0][i], B, d.H[i], d.W[i], p->ccatp[0][i]); src[ns].g.Cp = p->ccatp[0][i];
    src[ns].c_offset = off_same; src[ns].mode = MG_SEG_SAME; ++ns;
    if (i + 1 < n) {
      src[ns].g = grid_of(ws, p->dcat[0][i + 1], B, d.H[i + 1], d.W[i + 1], p->ccatp[0][i + 1]); src[ns].g.Cp = p->ccatp[0][i + 1];
      src[ns].c_offset = 0; src[ns].mode = MG_SEG_POOL; ++ns;
    }
    if (i > 0) {
      const int off_up = (i - 1 > 0 ? cpad(d.C_in[i - 2]) : 0) + cpad(d.C_in[i - 1]);
      src[ns].g = grid_of(ws, p->dcat[0][i - 1], B, d.H[i - 1], d.W[i - 1], p->ccatp[0][i - 1]); src[ns].g.Cp = p->ccatp[0][i - 1];
      src[ns].c_offset = off_up; src[ns].mode = MG_SEG_UP; ++ns;
    }
    if (d.residual) {   // CAddTable passes the masked gradient of the output to the shortcut; nn.Padding keeps its first C_in channels
      src[ns].g = grid_of(ws, p->D[L - 1][i], B, d.H[i], d.W[i], d.C_out[i]);
      src[ns].c_offset = 0; src[ns].mode = MG_SEG_SAME; ++ns;
    }
    mg_grid X = grid_of(ws, p->X[i], B, d.H[i], d.W[i], d.C_in[i]);
    mg_grid DX = grid_of(ws, p->DX[i], B, d.H[i], d.W[i], d.C_in[i]);
    MG_TRY(mg_grad_combine(ctx, &X, 0, nullptr, ns, src, &DX, nullptr));
    MG_TRY(mg_export_nchw(ctx, &DX, dx[i]));
  }
  return MG_OK;
}

}  // namespace

extern "C" {

int mg_stage_backward(mg_stage_plan* p, void* workspace, const float* const* dy, const mg_stage_params* prm, float* const* dx, float scale) {
  return stage_backward(p, workspace, dy, prm, dx, scale, true, "stage_backward");
}

int mg_stage_update_grad_input(mg_stage_plan* p, void* workspace, const float* const* dy, const mg_stage_params* prm, float* const* dx) {
  const int rc = stage_backward(p, workspace, dy, prm, dx, 0.f, false, "stage_update_grad_input");
  if (rc == MG_OK) p->grad_input_ready = 1;
  return rc;
}

int mg_stage_acc_grad_parameters(mg_stage_plan* p, void* workspace, const mg_stage_params* prm, float scale) {
  if (!p || !workspace || !prm) return MG_ERR_INVALID_ARG;
  mg_ctx* ctx = p->ctx;
  const mg_stage_desc& d = p->d;
  const int n = p->n, L = p->layers, B = p->batch;
  char* ws = (char*)workspace;
  MG_REQUIRE(ctx, p->grad_input_ready, MG_ERR_INVALID_ARG,
             "stage_acc_grad_parameters: no mg_stage_update_grad_input since the last mg_stage_forward of this plan");
  const bool frozen = p->last_training == 0;
  // every BatchNorm of the stage in one launch, from the sums, batch statistics and G the update phase left in the workspace
  mg_bn_param_job jobs[2 * MG_STAGE_MAX_GRIDS];
  memset(jobs, 0, sizeof(jobs));
  for (int l = 0; l < L; ++l)
    for (int i = 0; i < n; ++i) {
      const int k = l * n + i;
      MG_REQUIRE(ctx, prm->conv_gw[k] && prm->conv_gb[k] && prm->bn_gg[k] && prm->bn_gb[k], MG_ERR_INVALID_ARG,
                 "stage_acc_grad_parameters: gradient tensors of conv / BN %d are null", k);
      mg_bn_param_job& j = jobs[k];
      j.sums = (const mg_sum*)(ws + p->bsums[l][i]);
      j.count = (int64_t)B * d.H[i] * d.W[i];
      j.C = d.C_out[i];
      j.frozen = frozen ? 1 : 0;
      j.gamma = prm->bn_g[k];
      j.save_mean = (const float*)(ws + p->mean[l][i]); j.save_invstd = (const float*)(ws + p->invstd[l][i]);
      j.running_mean = prm->bn_rm[k]; j.running_var = prm->bn_rv[k];
      j.eps = d.eps;
      j.gscale = scale;
      j.dgamma = prm->bn_gg[k]; j.dbeta = prm->bn_gb[k]; j.conv_dbias = prm->conv_gb[k];
    }
  MG_TRY(mg_bn_param_grad(ctx, L * n, jobs));
  for (int l = L - 1; l >= 0; --l)
    for (int i = 0; i < n; ++i) {
      mg_conv_desc cd;
      make_desc(p, ws, l, i, &cd);
      mg_grid Gg = grid_of(ws, p->G[l][i], B, d.H[i], d.W[i], d.C_out[i]);
      MG_TRY(mg_conv_backward_weight(ctx, &cd, &Gg, prm->conv_gw[l * n + i], nullptr, scale));
    }
  return MG_OK;
}

}  // extern "C"
