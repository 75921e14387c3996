// C-ABI entry points: context management, conv dispatch (tcgen05 vs CUDA-core), data-parallel
// communicator.  See include/mgconv.h for the contract of every function.
#include "common.cuh"
#include "tma.cuh"
#include <dlfcn.h>
#include <stdlib.h>
#include <algorithm>
#include <new>

// simt_conv.cu
int simt_conv_forward(mg_ctx*, const mg_conv_desc*, const float*, const float*, mg_grid*, mg_sum*);
int simt_conv_backward_data(mg_ctx*, const mg_conv_desc*, const float*, const mg_grid*, mg_grid*);
int simt_strided_dgrad(mg_ctx*, const mg_conv_desc*, const float*, const mg_grid*, mg_grid*);
int simt_conv_backward_weight(mg_ctx*, const mg_conv_desc*, const mg_grid*, float*, float*, float);
// umma_conv.cu
bool umma_conv_supported(const mg_ctx*, const mg_conv_desc*, int kind);
size_t umma_packed_bytes(const mg_conv_desc*, int transposed);
int umma_pack_weights(mg_ctx*, const mg_conv_desc*, const float*, void*, int transposed);
int umma_pack_weights_batched(mg_ctx*, int n, const mg_conv_desc* const*, const float* const*, void* const*, const int32_t*);
int umma_conv_forward(mg_ctx*, const mg_conv_desc*, const void*, const float*, mg_grid*, mg_sum*);
int umma_conv_backward_data(mg_ctx*, const mg_conv_desc*, const void*, const mg_grid*, mg_grid*);
int umma_conv_backward_weight(mg_ctx*, const mg_conv_desc*, const mg_grid*, float*, float*, float);

#include <vector>
struct ProfState {
  std::vector<cudaEvent_t> pool;             // events, reused
  std::vector<std::pair<int, int>> spans;    // (begin, end) indices into pool
  size_t used = 0;
  double acc_ms = 0;                         // spans already folded
  int64_t launches = 0;
};

// fold the pending spans into acc_ms (synchronises the stream) so the pool can be reused
static void prof_flush(mg_ctx* ctx) {
  ProfState* ps = (ProfState*)ctx->prof;
  if (!ps || ps->spans.empty()) return;
  cudaStreamSynchronize(ctx->stream);
  for (auto& sp : ps->spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ps->pool[sp.first], ps->pool[sp.second]) == cudaSuccess) ps->acc_ms += ms;
  }
  ps->spans.clear();
  ps->used = 0;
}

struct ProfSpan {
  mg_ctx* ctx; int b = -1;
  explicit ProfSpan(mg_ctx* c) : ctx(c) {
    if (!c->profile) return;
    ProfState* ps = (ProfState*)c->prof;
    if (ps->used + 2 > 8192) prof_flush(c);
    while (ps->pool.size() < ps->used + 2) { cudaEvent_t e; cudaEventCreate(&e); ps->pool.push_back(e); }
    b = (int)ps->used; ps->used += 2;
    cudaEventRecord(ps->pool[b], c->stream);
  }
  ~ProfSpan() {
    if (b < 0) return;
    ProfState* ps = (ProfState*)ctx->prof;
    cudaEventRecord(ps->pool[b + 1], ctx->stream);
    ps->spans.push_back({b, b + 1});
    ps->launches++;
  }
};

static bool use_umma(const mg_ctx* ctx, const mg_conv_desc* d, const void* wpack, int kind) {
  if (ctx->dtype != MG_BF16 || ctx->impl == MG_IMPL_SIMT) return false;
  if (kind != 2 && !wpack) return false;
  return umma_conv_supported(ctx, d, kind);
}

extern "C" {

int mg_version(void) { return 100; }

int mg_ctx_create(int device, void* cuda_stream, int dtype, mg_ctx** out) {
  if (!out || (dtype != MG_F32 && dtype != MG_BF16)) return MG_ERR_INVALID_ARG;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return MG_ERR_CUDA;
  mg_ctx* c = new (std::nothrow) mg_ctx();
  if (!c) return MG_ERR_INVALID_ARG;
  memset(c, 0, sizeof(*c));
  c->device = device; c->stream = (cudaStream_t)cuda_stream; c->dtype = dtype; c->impl = MG_IMPL_AUTO;
  c->lane_stream[0] = c->stream;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return MG_ERR_CUDA; }
  if (prop.major != 10) {  // sm_100a only: no fallback architecture
    delete c;
    return MG_ERR_UNSUPPORTED;
  }
  c->num_sms = prop.multiProcessorCount;
  *out = c;
  return MG_OK;
}

int mg_ctx_profile(mg_ctx* ctx, int on) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  if (on && !ctx->prof) ctx->prof = new (std::nothrow) ProfState();
  if (on && !ctx->prof) return MG_ERR_INVALID_ARG;
  ctx->profile = on ? 1 : 0;
  return MG_OK;
}

int mg_ctx_profile_read(mg_ctx* ctx, double* conv_ms, int64_t* conv_launches) {
  if (!ctx || !conv_ms || !conv_launches) return MG_ERR_INVALID_ARG;
  ProfState* ps = (ProfState*)ctx->prof;
  if (!ps) { *conv_ms = 0; *conv_launches = 0; return MG_OK; }
  prof_flush(ctx);
  *conv_ms = ps->acc_ms; *conv_launches = ps->launches;
  ps->acc_ms = 0; ps->launches = 0;
  return MG_OK;
}

int mg_ctx_destroy(mg_ctx* ctx) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  if (ctx->prof) {
    ProfState* ps = (ProfState*)ctx->prof;
    for (auto e : ps->pool) cudaEventDestroy(e);
    delete ps;
  }
  mg_comm_destroy(ctx);
  if (ctx->ws) cudaFree(ctx->ws);
  for (int l = 1; l < MG_MAX_LANES; ++l) {
    if (ctx->lane_ws[l]) cudaFree(ctx->lane_ws[l]);
    if (ctx->lane_stream[l]) cudaStreamDestroy(ctx->lane_stream[l]);
  }
  for (int l = 0; l < MG_MAX_LANES; ++l) if (ctx->lane_ev[l]) cudaEventDestroy(ctx->lane_ev[l]);
  for (int l = 0; l < MG_MAX_LANES; ++l) if (ctx->up_ws[l]) cudaFree(ctx->up_ws[l]);
  for (int l = 0; l < MG_MAX_LANES; ++l) if (ctx->sum_scratch[l]) cudaFree(ctx->sum_scratch[l]);
  for (int e = 0; e < ctx->n_events; ++e) cudaEventDestroy(ctx->events[e]);
  free(ctx->events);
  if (ctx->pack_dev) cudaFree(ctx->pack_dev);
  free(ctx->pack_host);
  delete (TmapCache*)ctx->tmaps;
  delete ctx;
  return MG_OK;
}

int mg_ctx_set_stream(mg_ctx* ctx, void* s) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  ctx->lane_stream[0] = (cudaStream_t)s;
  ctx->stream = ctx->lane_stream[ctx->cur_lane];
  return MG_OK;
}

int mg_ctx_lane(mg_ctx* ctx, int lane) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, lane >= 0 && lane < MG_MAX_LANES, MG_ERR_INVALID_ARG, "lane %d out of range (0..%d)", lane, MG_MAX_LANES - 1);
  if (lane && !ctx->lane_stream[lane]) {
    MG_CUDA(ctx, cudaSetDevice(ctx->device));
    MG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->lane_stream[lane], cudaStreamNonBlocking));
  }
  ctx->cur_lane = lane;
  ctx->stream = ctx->lane_stream[lane];
  return MG_OK;
}

static int ensure_events(mg_ctx* ctx, int ev) {
  MG_REQUIRE(ctx, ev >= 0 && ev < (1 << 16), MG_ERR_INVALID_ARG, "event id %d", ev);
  if (ev >= ctx->n_events) {
    const int n = std::max(ev + 1, std::max(64, 2 * ctx->n_events));
    cudaEvent_t* p = (cudaEvent_t*)realloc(ctx->events, (size_t)n * sizeof(cudaEvent_t));
    MG_REQUIRE(ctx, p != nullptr, MG_ERR_INVALID_ARG, "events: out of memory");
    ctx->events = p;
    for (int e = ctx->n_events; e < n; ++e) MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->events[e], cudaEventDisableTiming));
    ctx->n_events = n;
  }
  return MG_OK;
}

int mg_ctx_event_record(mg_ctx* ctx, int ev) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  int rc = ensure_events(ctx, ev);
  if (rc) return rc;
  MG_CUDA(ctx, cudaEventRecord(ctx->events[ev], ctx->stream));
  return MG_OK;
}

int mg_ctx_event_wait(mg_ctx* ctx, int ev) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  int rc = ensure_events(ctx, ev);
  if (rc) return rc;
  MG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->events[ev], 0));
  return MG_OK;
}
int mg_ctx_set_impl(mg_ctx* ctx, int impl) {
  if (!ctx || impl < 0 || impl > 2) return MG_ERR_INVALID_ARG;
  ctx->impl = impl; return MG_OK;
}
int mg_ctx_set_tuning(mg_ctx* ctx, int knob, int value) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  if (knob == MG_TUNE_HALO_SUBTILES) { MG_REQUIRE(ctx, value >= 0 && value <= 2, MG_ERR_INVALID_ARG, "set_tuning: sub-tiles %d", value); ctx->tune_mt = value; return MG_OK; }
  if (knob == MG_TUNE_PERSISTENT) { MG_REQUIRE(ctx, value >= 0 && value <= 2, MG_ERR_INVALID_ARG, "set_tuning: persistent %d", value); ctx->tune_persist = value; return MG_OK; }
  if (knob == MG_TUNE_STEM_FUSED_STATS) { MG_REQUIRE(ctx, value >= 0 && value <= 1, MG_ERR_INVALID_ARG, "set_tuning: stem fused stats %d", value); ctx->tune_stem_fused = value; return MG_OK; }
  MG_FAIL(ctx, MG_ERR_INVALID_ARG, "set_tuning: unknown knob %d", knob);
}
int mg_ctx_sync(mg_ctx* ctx) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  for (int l = 0; l < MG_MAX_LANES; ++l)
    if (l == 0 || ctx->lane_stream[l]) MG_CUDA(ctx, cudaStreamSynchronize(ctx->lane_stream[l]));
  if (ctx->comm_stream) MG_CUDA(ctx, cudaStreamSynchronize(ctx->comm_stream));
  return MG_OK;
}
const char* mg_last_error(mg_ctx* ctx) { return ctx ? ctx->err : "null context"; }
int mg_ctx_tc_launch_count(mg_ctx* ctx, int64_t* out) { if (!ctx || !out) return MG_ERR_INVALID_ARG; *out = ctx->tc_launches; return MG_OK; }
int mg_ctx_launch_count(mg_ctx* ctx, int64_t* out) { if (!ctx || !out) return MG_ERR_INVALID_ARG; *out = ctx->launches; return MG_OK; }

// ---- conv dispatch ------------------------------------------------------------------
size_t mg_conv_packed_bytes(const mg_conv_desc* d, int transposed) { return d ? umma_packed_bytes(d, transposed) : 0; }

int mg_conv_pack_weights(mg_ctx* ctx, const mg_conv_desc* d, const float* w, void* wpack, int transposed) {
  if (!ctx || !d || !w || !wpack) return MG_ERR_INVALID_ARG;
  return umma_pack_weights(ctx, d, w, wpack, transposed);
}

int mg_conv_pack_weights_batched(mg_ctx* ctx, int32_t n, const mg_conv_desc* const* descs, const float* const* w, void* const* wpack,
                                 const int32_t* transposed) {
  if (!ctx || n < 0 || (n && (!descs || !w || !wpack || !transposed))) return MG_ERR_INVALID_ARG;
  if (n == 0) return MG_OK;
  return umma_pack_weights_batched(ctx, n, descs, w, wpack, transposed);
}

int mg_conv_forward(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const void* wpack, const float* bias,
                    mg_grid* y, mg_sum* bn_sums) {
  if (!ctx || !d || !y || !y->data) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, y->C == d->Cout && y->Cp >= y->C && y->Cp % 8 == 0, MG_ERR_SHAPE, "conv_forward: y.C %d Cp %d vs Cout %d", y->C, y->Cp, d->Cout);
  int Ho = (d->H + 2 * d->pad - d->ksize) / d->stride + 1, Wo = (d->W + 2 * d->pad - d->ksize) / d->stride + 1;
  MG_REQUIRE(ctx, y->H == Ho && y->W == Wo && y->N == d->seg[0].N, MG_ERR_SHAPE, "conv_forward: y is %dx%d, expected %dx%d", y->H, y->W, Ho, Wo);
  ProfSpan span(ctx);
  if (use_umma(ctx, d, wpack, 0)) return umma_conv_forward(ctx, d, wpack, bias, y, bn_sums);
  MG_REQUIRE(ctx, ctx->impl != MG_IMPL_TCGEN05, MG_ERR_UNSUPPORTED, "conv_forward: shape not supported by the tcgen05 path");
  MG_REQUIRE(ctx, w != nullptr, MG_ERR_INVALID_ARG, "conv_forward: null weights");
  return simt_conv_forward(ctx, d, w, bias, y, bn_sums);
}

int mg_conv_backward_data(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const void* wpack_t, const mg_grid* g, mg_grid* dcat) {
  if (!ctx || !d || !g || !dcat) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, g->C == d->Cout, MG_ERR_SHAPE, "conv_backward_data: g.C %d != Cout %d", g->C, d->Cout);
  MG_REQUIRE(ctx, dcat->H == d->H && dcat->W == d->W && dcat->N == g->N, MG_ERR_SHAPE, "conv_backward_data: dcat shape");
  ProfSpan span(ctx);
  if (d->stride != 1) {   // the image-fed strided stem: a CUDA-core kernel in every dtype and impl (simt_conv.cu: stem_dgrad_kernel)
    MG_REQUIRE(ctx, w != nullptr, MG_ERR_INVALID_ARG, "conv_backward_data: null weights");
    return simt_strided_dgrad(ctx, d, w, g, dcat);
  }
  if (use_umma(ctx, d, wpack_t, 1)) return umma_conv_backward_data(ctx, d, wpack_t, g, dcat);
  MG_REQUIRE(ctx, ctx->impl != MG_IMPL_TCGEN05, MG_ERR_UNSUPPORTED, "conv_backward_data: shape not supported by the tcgen05 path");
  MG_REQUIRE(ctx, w != nullptr, MG_ERR_INVALID_ARG, "conv_backward_data: null weights");
  return simt_conv_backward_data(ctx, d, w, g, dcat);
}

int mg_conv_backward_weight(mg_ctx* ctx, const mg_conv_desc* d, const mg_grid* g, float* dw, float* dbias, float gscale) {
  if (!ctx || !d || !g || !dw) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, g->C == d->Cout, MG_ERR_SHAPE, "conv_backward_weight: g.C %d != Cout %d", g->C, d->Cout);
  ProfSpan span(ctx);
  if (use_umma(ctx, d, nullptr, 2)) return umma_conv_backward_weight(ctx, d, g, dw, dbias, gscale);
  MG_REQUIRE(ctx, ctx->impl != MG_IMPL_TCGEN05, MG_ERR_UNSUPPORTED, "conv_backward_weight: shape not supported by the tcgen05 path");
  return simt_conv_backward_weight(ctx, d, g, dw, dbias, gscale);
}

// ---- data parallel: NCCL resolved at run time from the process (torch bundles libnccl.so.2)
typedef struct { char internal[128]; } mg_nccl_uid;
typedef int (*fn_ncclGetUniqueId)(mg_nccl_uid*);
typedef int (*fn_ncclCommInitRank)(void**, int, mg_nccl_uid, int);
typedef int (*fn_ncclCommDestroy)(void*);
typedef int (*fn_ncclAllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*fn_ncclGetErrorString)(int);

static struct {
  void* h;
  fn_ncclGetUniqueId GetUniqueId;
  fn_ncclCommInitRank CommInitRank;
  fn_ncclCommDestroy CommDestroy;
  fn_ncclAllReduce AllReduce;
  fn_ncclGetErrorString GetErrorString;
} g_nccl;

static int load_nccl() {
  if (g_nccl.h) return 0;
  const char* names[] = {getenv("MGCONV_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) { if (n && (h = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break; }
  if (!h) return -1;
  g_nccl.GetUniqueId = (fn_ncclGetUniqueId)dlsym(h, "ncclGetUniqueId");
  g_nccl.CommInitRank = (fn_ncclCommInitRank)dlsym(h, "ncclCommInitRank");
  g_nccl.CommDestroy = (fn_ncclCommDestroy)dlsym(h, "ncclCommDestroy");
  g_nccl.AllReduce = (fn_ncclAllReduce)dlsym(h, "ncclAllReduce");
  g_nccl.GetErrorString = (fn_ncclGetErrorString)dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllReduce) return -1;
  g_nccl.h = h;
  return 0;
}

#define MG_NCCL(ctx, expr)                                                                  \
  do {                                                                                      \
    int _r = (expr);                                                                        \
    if (_r != 0) MG_FAIL(ctx, MG_ERR_NCCL, "%s: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "nccl error"); \
  } while (0)

int mg_comm_unique_id(void* out128) {
  if (!out128 || load_nccl()) return MG_ERR_NCCL;
  return g_nccl.GetUniqueId((mg_nccl_uid*)out128) == 0 ? MG_OK : MG_ERR_NCCL;
}

int mg_comm_init(mg_ctx* ctx, int rank, int nranks, const void* id128) {
  if (!ctx || !id128 || rank < 0 || rank >= nranks) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, load_nccl() == 0, MG_ERR_NCCL, "cannot load libnccl.so.2 (set MGCONV_NCCL_LIB)");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  mg_nccl_uid uid; memcpy(&uid, id128, sizeof(uid));
  MG_NCCL(ctx, g_nccl.CommInitRank(&ctx->nccl_comm, nranks, uid, rank));
  MG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->comm_stream, cudaStreamNonBlocking));
  MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_compute, cudaEventDisableTiming));
  MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_comm, cudaEventDisableTiming));
  ctx->rank = rank; ctx->nranks = nranks;
  return MG_OK;
}

// The communicator outlives the per-shape plans: a host keeps ONE owner context per device (mg_comm_init once) and lends its
// communicator to every working context (a new one whenever the input shape changes -- the partial last batch of
// pipelines/standard/test.lua:40-44).  The borrower gets its own communication stream and events.
int mg_comm_share(mg_ctx* ctx, const mg_ctx* owner) {
  if (!ctx || !owner) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, owner->nccl_comm != nullptr, MG_ERR_NCCL, "comm_share: the owner has no communicator (mg_comm_init it first)");
  MG_REQUIRE(ctx, owner->device == ctx->device, MG_ERR_INVALID_ARG, "comm_share: owner on device %d, context on %d", owner->device, ctx->device);
  if (ctx->nccl_comm == owner->nccl_comm) return MG_OK;
  MG_REQUIRE(ctx, ctx->nccl_comm == nullptr, MG_ERR_INVALID_ARG, "comm_share: the context already has a communicator");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  MG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->comm_stream, cudaStreamNonBlocking));
  MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_compute, cudaEventDisableTiming));
  MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_comm, cudaEventDisableTiming));
  ctx->nccl_comm = owner->nccl_comm; ctx->comm_borrowed = 1;
  ctx->rank = owner->rank; ctx->nranks = owner->nranks;
  return MG_OK;
}

int mg_comm_destroy(mg_ctx* ctx) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  if (ctx->nccl_comm && !ctx->comm_borrowed) g_nccl.CommDestroy(ctx->nccl_comm);
  ctx->nccl_comm = nullptr; ctx->comm_borrowed = 0;
  if (ctx->comm_stream) { cudaStreamDestroy(ctx->comm_stream); ctx->comm_stream = nullptr; }
  if (ctx->ev_compute) { cudaEventDestroy(ctx->ev_compute); ctx->ev_compute = nullptr; }
  if (ctx->ev_comm) { cudaEventDestroy(ctx->ev_comm); ctx->ev_comm = nullptr; }
  return MG_OK;
}

int mg_allreduce_launch(mg_ctx* ctx, void* buf, int64_t count, int is_double) {
  if (!ctx || !buf || count < 0) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, ctx->nccl_comm != nullptr, MG_ERR_NCCL, "allreduce: communicator not initialised");
  // comm stream waits for everything enqueued so far on the compute stream (the bucket's wgrads) -- on EVERY lane: the
  // gradients of one bucket come from chains that ran on different lanes
  MG_CUDA(ctx, cudaEventRecord(ctx->ev_compute, ctx->stream));
  MG_CUDA(ctx, cudaStreamWaitEvent(ctx->comm_stream, ctx->ev_compute, 0));
  for (int l = 0; l < MG_MAX_LANES; ++l) {
    if (l == ctx->cur_lane || (l && !ctx->lane_stream[l])) continue;
    if (!ctx->lane_ev[l]) MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->lane_ev[l], cudaEventDisableTiming));
    MG_CUDA(ctx, cudaEventRecord(ctx->lane_ev[l], ctx->lane_stream[l]));
    MG_CUDA(ctx, cudaStreamWaitEvent(ctx->comm_stream, ctx->lane_ev[l], 0));
  }
  const int ncclInt64 = 4, ncclFloat32 = 7, ncclFloat64 = 8, ncclSum = 0;
  MG_NCCL(ctx, g_nccl.AllReduce(buf, buf, (size_t)count, is_double == 2 ? ncclInt64 : (is_double ? ncclFloat64 : ncclFloat32), ncclSum, ctx->nccl_comm, ctx->comm_stream));
  return MG_OK;
}

int mg_allreduce_inline(mg_ctx* ctx, void* buf, int64_t count, int is_double) {
  if (!ctx || !buf || count < 0) return MG_ERR_INVALID_ARG;
  MG_REQUIRE(ctx, ctx->nccl_comm != nullptr, MG_ERR_NCCL, "allreduce: communicator not initialised");
  const int ncclInt64 = 4, ncclFloat32 = 7, ncclFloat64 = 8, ncclSum = 0;
  MG_NCCL(ctx, g_nccl.AllReduce(buf, buf, (size_t)count, is_double == 2 ? ncclInt64 : (is_double ? ncclFloat64 : ncclFloat32), ncclSum, ctx->nccl_comm, ctx->stream));
  return MG_OK;
}

int mg_allreduce_wait(mg_ctx* ctx) {
  if (!ctx) return MG_ERR_INVALID_ARG;
  if (!ctx->nccl_comm) return MG_OK;
  MG_CUDA(ctx, cudaEventRecord(ctx->ev_comm, ctx->comm_stream));
  MG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_comm, 0));
  return MG_OK;
}

}  // extern "C"
