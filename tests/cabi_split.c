/* Pure-C driver of the split plan-level backward (include/mgconv.h): on one residual multigrid unit,
 *   mg_stage_forward -> mg_stage_update_grad_input -> mg_stage_acc_grad_parameters(scale)
 * must leave the bits of
 *   mg_stage_forward -> mg_stage_backward(scale)
 * in the input gradients, every parameter gradient and the running statistics, in training and in evaluation mode; the update
 * half alone must leave the parameter gradients untouched, and the accumulate half must fail without an update since the last
 * forward.  The problem is generated here (fixed LCG), so the driver needs no input file.
 *
 *   tests/cabi_split <bf16|fp32> <scale>      prints "cabi_split ok" and exits 0 when everything holds
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>
#include <cuda_runtime_api.h>
#include "mgconv.h"

#define CHECK_CUDA(e) do { cudaError_t _e = (e); if (_e != cudaSuccess) { fprintf(stderr, "CUDA error %s at %s:%d\n", cudaGetErrorString(_e), __FILE__, __LINE__); exit(2); } } while (0)
#define CHECK_MG(ctx, e) do { int _r = (e); if (_r != 0) { fprintf(stderr, "mgconv status %d at %s:%d: %s\n", _r, __FILE__, __LINE__, mg_last_error(ctx)); exit(3); } } while (0)

#define NT (2 * MG_STAGE_MAX_GRIDS)

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static float uniform(float lo, float hi) {
  rng_state = rng_state * 6364136223846793005ull + 1442695040888963407ull;
  return lo + (hi - lo) * (float)((rng_state >> 40) * (1.0 / 16777216.0));
}
static float* dev_random(size_t n, float lo, float hi, float** host) {
  float* h = (float*)malloc(n * sizeof(float));
  float* d = NULL;
  for (size_t i = 0; i < n; ++i) h[i] = uniform(lo, hi);
  CHECK_CUDA(cudaMalloc((void**)&d, n * sizeof(float)));
  CHECK_CUDA(cudaMemcpy(d, h, n * sizeof(float), cudaMemcpyHostToDevice));
  *host = h;
  return d;
}
static void dev_fill(float* d, const float* h, size_t n) { CHECK_CUDA(cudaMemcpy(d, h, n * sizeof(float), cudaMemcpyHostToDevice)); }
static float* dev_const(size_t n, float v) {
  float* h = (float*)malloc(n * sizeof(float));
  float* d = NULL;
  for (size_t i = 0; i < n; ++i) h[i] = v;
  CHECK_CUDA(cudaMalloc((void**)&d, n * sizeof(float)));
  dev_fill(d, h, n);
  free(h);
  return d;
}
static float* download(const float* d, size_t n) {
  float* h = (float*)malloc(n * sizeof(float));
  CHECK_CUDA(cudaMemcpy(h, d, n * sizeof(float), cudaMemcpyDeviceToHost));
  return h;
}

typedef struct {   /* everything a run leaves behind, on the host */
  float* dx[MG_STAGE_MAX_GRIDS];
  float* t[NT][6];   /* conv_gw, conv_gb, bn_gg, bn_gb, bn_rm, bn_rv */
} result;

static int n, L, batch;
static mg_stage_desc d;
static size_t nx[MG_STAGE_MAX_GRIDS], ny[MG_STAGE_MAX_GRIDS], nw[NT], nc[NT];
static float* h_rm[NT]; static float* h_rv[NT];
static const float SENTINEL = 0.375f;

static void reset(mg_stage_params* prm) {   /* running statistics to their initial values, gradients to the sentinel */
  for (int k = 0; k < L * n; ++k) {
    float* h = (float*)malloc(nw[k] * sizeof(float));
    for (size_t i = 0; i < nw[k]; ++i) h[i] = SENTINEL;
    dev_fill(prm->conv_gw[k], h, nw[k]); dev_fill(prm->conv_gb[k], h, nc[k]); dev_fill(prm->bn_gg[k], h, nc[k]); dev_fill(prm->bn_gb[k], h, nc[k]);
    free(h);
    dev_fill(prm->bn_rm[k], h_rm[k], nc[k]); dev_fill(prm->bn_rv[k], h_rv[k], nc[k]);
  }
}
static void collect(const mg_stage_params* prm, float* const* dx, result* r) {
  CHECK_CUDA(cudaDeviceSynchronize());
  for (int i = 0; i < n; ++i) r->dx[i] = download(dx[i], nx[i]);
  for (int k = 0; k < L * n; ++k) {
    r->t[k][0] = download(prm->conv_gw[k], nw[k]); r->t[k][1] = download(prm->conv_gb[k], nc[k]);
    r->t[k][2] = download(prm->bn_gg[k], nc[k]);   r->t[k][3] = download(prm->bn_gb[k], nc[k]);
    r->t[k][4] = download(prm->bn_rm[k], nc[k]);   r->t[k][5] = download(prm->bn_rv[k], nc[k]);
  }
}
static int same(const result* a, const result* b, const char* what) {
  static const char* names[6] = {"conv gradWeight", "conv gradBias", "bn gradWeight", "bn gradBias", "running_mean", "running_var"};
  for (int i = 0; i < n; ++i)
    if (memcmp(a->dx[i], b->dx[i], nx[i] * sizeof(float))) { fprintf(stderr, "%s: gradInput of grid %d differs\n", what, i); return 0; }
  for (int k = 0; k < L * n; ++k)
    for (int f = 0; f < 6; ++f) {
      const size_t m = f == 0 ? nw[k] : nc[k];
      if (memcmp(a->t[k][f], b->t[k][f], m * sizeof(float))) { fprintf(stderr, "%s: %s of layer %d differs\n", what, names[f], k); return 0; }
    }
  return 1;
}

int main(int argc, char** argv) {
  if (argc != 3) { fprintf(stderr, "usage: %s <bf16|fp32> <scale>\n", argv[0]); return 1; }
  const int dtype = strcmp(argv[1], "bf16") == 0 ? MG_BF16 : MG_F32;
  const float scale = (float)atof(argv[2]);
  /* three grids, 13 channels on the finest (not a multiple of 8), a padded shortcut (C_in < C_out) */
  const int cin[3] = {13, 16, 8}, cout[3] = {21, 16, 8}, hw[3] = {16, 8, 4};
  memset(&d, 0, sizeof(d));
  d.n_scales = n = 3; d.residual = 1; d.eps = 1e-5f; d.momentum = 0.1f;
  batch = 3; L = 2;
  for (int i = 0; i < n; ++i) { d.C_in[i] = cin[i]; d.C_out[i] = cout[i]; d.H[i] = d.W[i] = hw[i]; d.ksize[i] = 3; }

  cudaStream_t stream;
  CHECK_CUDA(cudaStreamCreate(&stream));
  mg_ctx* ctx = NULL;
  if (mg_ctx_create(0, (void*)stream, dtype, &ctx) != 0) { fprintf(stderr, "mg_ctx_create failed (no sm_100 GPU?)\n"); return 3; }

  const float* x[MG_STAGE_MAX_GRIDS]; const float* dy[MG_STAGE_MAX_GRIDS];
  float* y[MG_STAGE_MAX_GRIDS]; float* dx[MG_STAGE_MAX_GRIDS];
  float* scratch;
  for (int i = 0; i < n; ++i) {
    nx[i] = (size_t)batch * d.C_in[i] * d.H[i] * d.W[i];
    ny[i] = (size_t)batch * d.C_out[i] * d.H[i] * d.W[i];
    x[i] = dev_random(nx[i], -1.f, 1.f, &scratch); free(scratch);
    dy[i] = dev_random(ny[i], -1.f, 1.f, &scratch); free(scratch);
    y[i] = dev_const(ny[i], 0.f); dx[i] = dev_const(nx[i], 0.f);
  }
  mg_stage_params prm;
  memset(&prm, 0, sizeof(prm));
  for (int l = 0; l < L; ++l)
    for (int i = 0; i < n; ++i) {
      const int k = l * n + i;
      int ccat = (l == 0 ? d.C_in[i] : d.C_out[i]);
      if (i > 0) ccat += (l == 0 ? d.C_in[i - 1] : d.C_out[i - 1]);
      if (i + 1 < n) ccat += (l == 0 ? d.C_in[i + 1] : d.C_out[i + 1]);
      nc[k] = (size_t)d.C_out[i];
      nw[k] = nc[k] * ccat * 9;
      prm.conv_w[k] = dev_random(nw[k], -0.2f, 0.2f, &scratch); free(scratch);
      prm.conv_b[k] = dev_random(nc[k], -0.1f, 0.1f, &scratch); free(scratch);
      prm.bn_g[k] = dev_random(nc[k], 0.5f, 1.5f, &scratch); free(scratch);
      prm.bn_b[k] = dev_random(nc[k], -0.2f, 0.2f, &scratch); free(scratch);
      prm.bn_rm[k] = dev_random(nc[k], -0.2f, 0.2f, &h_rm[k]);
      prm.bn_rv[k] = dev_random(nc[k], 0.5f, 2.0f, &h_rv[k]);
      prm.conv_gw[k] = dev_const(nw[k], 0.f); prm.conv_gb[k] = dev_const(nc[k], 0.f);
      prm.bn_gg[k] = dev_const(nc[k], 0.f); prm.bn_gb[k] = dev_const(nc[k], 0.f);
    }
  mg_stage_plan* plan = NULL;
  CHECK_MG(ctx, mg_plan_create(ctx, &d, batch, &plan));
  void* ws = NULL;
  CHECK_CUDA(cudaMalloc(&ws, mg_plan_workspace_bytes(plan)));

  for (int training = 1; training >= 0; --training) {
    const char* mode = training ? "training" : "evaluation";
    result fused, upd, split;
    reset(&prm);
    CHECK_MG(ctx, mg_stage_forward(plan, ws, x, &prm, y, training));
    CHECK_MG(ctx, mg_stage_backward(plan, ws, dy, &prm, dx, scale));
    collect(&prm, dx, &fused);

    reset(&prm);
    for (int i = 0; i < n; ++i) CHECK_CUDA(cudaMemset(dx[i], 0, nx[i] * sizeof(float)));
    CHECK_MG(ctx, mg_stage_forward(plan, ws, x, &prm, y, training));
    int64_t tc0 = 0, tc1 = 0;
    mg_ctx_tc_launch_count(ctx, &tc0);
    CHECK_MG(ctx, mg_stage_update_grad_input(plan, ws, dy, &prm, dx));
    mg_ctx_tc_launch_count(ctx, &tc1);
    collect(&prm, dx, &upd);
    for (int k = 0; k < L * n; ++k)
      for (int f = 0; f < 4; ++f)
        for (size_t i = 0; i < (f == 0 ? nw[k] : nc[k]); ++i)
          if (upd.t[k][f][i] != SENTINEL) { fprintf(stderr, "%s: update_grad_input wrote parameter gradient %d of layer %d\n", mode, f, k); return 6; }
    CHECK_MG(ctx, mg_stage_acc_grad_parameters(plan, ws, &prm, scale));
    collect(&prm, dx, &split);
    if (!same(&fused, &split, mode)) return 7;

    /* a new forward invalidates what the update recorded */
    CHECK_MG(ctx, mg_stage_forward(plan, ws, x, &prm, y, training));
    if (mg_stage_acc_grad_parameters(plan, ws, &prm, scale) == 0) { fprintf(stderr, "%s: acc_grad_parameters after a new forward did not fail\n", mode); return 8; }
    printf("%s: split == fused, update phase %lld tcgen05 launches\n", mode, (long long)(tc1 - tc0));
  }
  mg_plan_destroy(plan);
  mg_ctx_destroy(ctx);
  printf("cabi_split ok\n");
  return 0;
}
