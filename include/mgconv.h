/* mgconv.h -- C ABI of the B200-native multigrid-convolution hot path.
 *
 * Drop-in boundary for buttomnutstoast/Multigrid-Neural-Architectures: every entry point
 * below replaces a chain of upstream Torch7 nn/cunn/cudnn module calls that the
 * reference's model builders assemble (the reference has no FFI of its own for this
 * path -- it is 100 % Lua on top of un-vendored luarocks packages -- so the "reference
 * interface" cited per function is the Lua builder code whose GPU work the call subsumes).
 *
 * Plain C, handle based, no C++ types or exceptions cross the boundary.  The header is
 * consumed verbatim by LuaJIT `ffi.cdef` (lua/mgconv_ffi.lua) and by Python ctypes/cffi
 * (mgconv/ffi.py).  Every function returns mg_status (0 = ok); the message of the last
 * failure on a context is available from mg_last_error().  The host (Torch) owns every tensor it
 * can see -- activations at the boundary, parameters, gradients, running statistics, stage workspaces --
 * and passes raw device pointers on every call (getParameters() re-homes weights after construction,
 * pipelines/standard/train.lua:115).  A context owns only small internal scratch, allocated lazily and
 * grown on demand (split weight-gradient partial sums per lane, the job table of the batched weight
 * packing, a few KB of deterministic-sum scratch, tensor-map cache) plus the NCCL communicator and its
 * streams / events; none of it is ever visible to or serialised by the host.
 * All work is enqueued on the stream given to the context; no call synchronises.
 *
 * Tensor convention ("grid"): NHWC, element type = the context dtype (fp32 or bf16),
 * channel pitch Cp = C rounded up to a multiple of 8, pad channels are zero.  A grid may
 * carry a *pending* per-channel affine (+ReLU) -- the BatchNorm(+ReLU) of its producer,
 * which is applied on the fly by whatever consumes the grid and never materialised:
 *      a[n,y,x,c] = relu?( scale[c] * data[n,y,x,c] + shift[c] )
 */
#ifndef MGCONV_H
#define MGCONV_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  MG_MAX_SEG = 6, /* input segments of one conv (3 for mg-conv; up to 6 after nn.ConcatUnet) */
  MG_MAX_SRC = 8  /* gradient contributions combined into one tensor */
};

typedef struct mg_ctx mg_ctx;

typedef enum {
  MG_OK = 0,
  MG_ERR_INVALID_ARG = 1,
  MG_ERR_SHAPE = 2,
  MG_ERR_CUDA = 3,
  MG_ERR_NCCL = 4,
  MG_ERR_UNSUPPORTED = 5
} mg_status;

typedef enum { MG_F32 = 0, MG_BF16 = 1 } mg_dtype;

/* how a source grid enters a conv's channel-concatenated input
 * (ResampleConcat, models/ilsvrc/rnmg.lua:41-89) */
typedef enum {
  MG_SEG_SAME = 0, /* nn.SelectTable(i)                                  rnmg.lua:64  */
  MG_SEG_POOL = 1, /* finer grid through SpatialMaxPooling(2,2,2,2):ceil rnmg.lua:54-60 */
  MG_SEG_UP = 2    /* coarser grid through SpatialUpSamplingNearest(2)   rnmg.lua:70-76 */
} mg_seg_mode;

typedef enum { MG_IMPL_AUTO = 0, MG_IMPL_SIMT = 1, MG_IMPL_TCGEN05 = 2 } mg_impl;

/* Per-channel sums behind BatchNorm (forward: sum y, sum y^2; backward: sum d, sum d*y) are accumulated DETERMINISTICALLY:
 * two's-complement fixed point in two 64-bit limbs, value = hi * 2^-10 + lo * 2^-54 (lo holds the 44 fractional bits of the
 * 2^-10 quantum of every contribution, with headroom for 2^19 contributions).  Every contribution is converted to this form
 * and added with integer atomics; integer addition is associative, so the totals are bit-identical from run to run, for any
 * order in which CTAs (or ranks: an int64 sum all-reduce) arrive.  Contributions must be below 2^40 in magnitude.
 * A buffer of n sums is n mg_sum (16 bytes each), zeroed by the caller before the first contribution. */
typedef struct { int64_t hi, lo; } mg_sum;

typedef struct {
  void* data;         /* device, NHWC [N][H][W][Cp] */
  const float* scale; /* device [Cp] or NULL (identity) */
  const float* shift; /* device [Cp] or NULL */
  int32_t relu;       /* ReLU after the affine */
  int32_t N, H, W, C, Cp;
} mg_grid;

/* One convolution of an mg stage: y = conv_k( cat_C[ seg_0 | seg_1 | ... ] ) + bias,
 * stride `stride` (1 everywhere except the ImageNet stem), zero padding `pad`.
 * Replaces Concat{Max,Select,UpSample} -> JoinTable(2) -> cudnn.SpatialConvolution
 * (models/ilsvrc/rnmg.lua:53-82 + 26/36; models/cifar/nmg.lua:46-79 + 22). */
typedef struct {
  int32_t n_seg;
  mg_grid seg[MG_MAX_SEG];
  int32_t seg_mode[MG_MAX_SEG];
  int32_t ksize, stride, pad;
  int32_t Cout;
  int32_t H, W; /* spatial size of the concatenated input (= output size when stride 1) */
  /* kernel variant of the 3x3 tensor-core path for mg_conv_forward / mg_conv_backward_data: 0 = heuristic,
   * MG_ALGO_*.  Hosts pick it by timing the variants once per layer -- what cudnn.benchmark = true does for the
   * reference's cudnn.SpatialConvolution (models/ilsvrc/rnmg.lua:230-231).  Every variant accumulates in the same
   * order, so the choice never changes results. */
  int32_t algo_fwd, algo_bwd_data;
} mg_conv_desc;
enum { MG_ALGO_AUTO = 0, MG_ALGO_TILE128 = 1, /* one 128-slot tile per CTA, several CTAs per SM */
       MG_ALGO_TILE256 = 2,                   /* two sub-tiles per CTA share every weight stage */
       MG_ALGO_RESIDENT = 3,                  /* persistent CTAs, whole weight image resident in shared memory */
       MG_ALGO_TILE128_DEEP = 4,              /* TILE128 with two CTAs per SM: two halo buffers, deeper weight ring */
       MG_ALGO_TILE256_DEEP = 5,              /* TILE256 with one CTA per SM: two halo buffers, deepest weight ring */
       MG_ALGO_TILE128_MID = 6,               /* TILE128 with three CTAs per SM (72 KB each) */
       MG_ALGO_PAIR128 = 7,                   /* tcgen05 CTA pairs (cta_group::2, M = 256 per MMA): each SM streams half of every weight stage */
       MG_ALGO_PAIR256 = 8,                   /* CTA pairs with two sub-tiles per CTA (512 slots per pair) */
       MG_ALGO_RESIDENT_PAIR = 9 };           /* persistent CTA pairs: half of the weight image resident per CTA, deeper halo ring */

typedef struct {
  mg_grid g;        /* gradient tensor of a consumer */
  int32_t c_offset; /* first channel of g that belongs to this tensor */
  int32_t mode;     /* MG_SEG_SAME: same resolution; MG_SEG_POOL: the consumer max-pooled this
                       tensor (g is at the coarser size, route through the 2x2 argmax);
                       MG_SEG_UP: the consumer upsampled this tensor (g is finer, sum 2x2);
                       3 = the consumer applied SpatialMaxPooling(3,3,2,2,1,1) (stem) */
  const void* aux;  /* mode 3: arg-max codes (uint8 [N][Ho][Wo][Cp], ky*3+kx) written by
                       mg_pool3s2_forward, or NULL to recompute the arg-max from x */
} mg_grad_src;

/* ---- context ------------------------------------------------------------------------ */
int mg_ctx_create(int device, void* cuda_stream, int dtype, mg_ctx** out);
int mg_ctx_destroy(mg_ctx* ctx);
int mg_ctx_set_stream(mg_ctx* ctx, void* cuda_stream);
int mg_ctx_set_impl(mg_ctx* ctx, int impl);          /* mg_impl; AUTO = tcgen05 for bf16 */
/* Lanes: the per-scale chains of an mg stage (conv -> BN -> ReLU on each grid, models/ilsvrc/rnmg.lua:91-159) are
 * independent until the next ResampleConcat, so a host may enqueue them on different lanes and let small grids
 * fill the tail of large ones.  Lane 0 is the stream given to mg_ctx_create / mg_ctx_set_stream, lanes 1..3 are
 * side streams owned by the context (each with its own scratch).  mg_ctx_lane selects the lane for the calls
 * that follow; ordering BETWEEN lanes is the host's job: mg_ctx_event_record(ev) marks a point on the current
 * lane, mg_ctx_event_wait(ev) makes the current lane wait for it (cudaEventRecord / cudaStreamWaitEvent). */
int mg_ctx_lane(mg_ctx* ctx, int lane);
int mg_ctx_event_record(mg_ctx* ctx, int ev);
int mg_ctx_event_wait(mg_ctx* ctx, int ev);
int mg_ctx_sync(mg_ctx* ctx);                         /* cutorch.synchronize() equivalent */
/* kernel-selection overrides for tests and tuning (the analogue of cudnn.benchmark / cudnn.fastest,
 * models/ilsvrc/rnmg.lua:230-231); value 0 = automatic choice */
enum { MG_TUNE_HALO_SUBTILES = 0, /* 1 / 2: 128-slot sub-tiles per CTA of the 3x3 tensor-core kernel */
       MG_TUNE_PERSISTENT = 1,    /* 1: weight-resident persistent kernel whenever the weights fit, 2: never */
       MG_TUNE_STEM_FUSED_STATS = 2 /* 1: the 7x7 stem kernel reduces the BatchNorm sums in its epilogue, 0: separate pass (default) */ };
int mg_ctx_set_tuning(mg_ctx* ctx, int knob, int value);
const char* mg_last_error(mg_ctx* ctx);
int mg_version(void);
int mg_ctx_launch_count(mg_ctx* ctx, int64_t* out);   /* kernels launched through this ctx */
int mg_ctx_tc_launch_count(mg_ctx* ctx, int64_t* out); /* ... of which tcgen05 tensor-core kernels */
/* CUDA-event timing of the convolution entry points (forward / backward_data / backward_weight):
 * while on, every such call is bracketed by two events on the context stream; read returns the
 * summed device time and the number of calls since the last read (synchronises the stream) */
int mg_ctx_profile(mg_ctx* ctx, int on);
int mg_ctx_profile_read(mg_ctx* ctx, double* conv_ms, int64_t* conv_calls);

/* ---- layout conversion at the Torch boundary (NCHW fp32 <-> grid) --------------------- */
int mg_import_nchw(mg_ctx* ctx, const float* src, mg_grid* dst);            /* put2GPU output -> grid */
int mg_export_nchw(mg_ctx* ctx, const mg_grid* src, float* dst);            /* applies pending affine */

/* GPU side of the data hooks (dataset/cifar100-whitened/donkey.lua:57-71 random crop, 131-139 horizontal flip with
 * probability 0.5, 19-23 of dataset/mnist-spt/donkey.lua mean / std normalisation; test hook: centre crop padded with zeros,
 * 166-175), applied to a batch that put2GPU (utils/utilfuncs.lua:3-30) already moved to the device:
 *   dst[n][c][y][x] = (src[n][c][y0[n]+y][x0[n] + (flip[n] ? oW-1-x : x)] - mean[c]) / std[c],   0 outside the source image.
 * src NCHW fp32 [N][C][H][W], dst NCHW fp32 [N][C][oH][oW]; y0 / x0 / flip (int32 [N]) and mean / std (fp32 [C]) are device
 * pointers and may be NULL (no offset / no flip / no normalisation). */
int mg_crop_flip_normalize(mg_ctx* ctx, const float* src, int32_t N, int32_t C, int32_t H, int32_t W, float* dst, int32_t oH, int32_t oW,
                           const int32_t* y0, const int32_t* x0, const int32_t* flip, const float* mean, const float* stdv);

/* ---- forward -------------------------------------------------------------------------- */
/* packed weight bytes for the tcgen05 path (0 when the SIMT path is used) */
size_t mg_conv_packed_bytes(const mg_conv_desc* d, int transposed);
/* repack fp32 [Cout][Ccat][k][k] master weights (cudnn.SpatialConvolution.weight) into the
 * UMMA operand images for forward (transposed=0) and dgrad (transposed=1) */
int mg_conv_pack_weights(mg_ctx* ctx, const mg_conv_desc* d, const float* w, void* wpack, int transposed);
/* the same for n (convolution, direction) pairs in ONE kernel launch: what a training step does for every
 * cudnn.SpatialConvolution of the model after optim.sgd changed the weights (models/basic_model.lua:64-66) */
int mg_conv_pack_weights_batched(mg_ctx* ctx, int32_t n, const mg_conv_desc* const* descs, const float* const* w,
                                 void* const* wpack, const int32_t* transposed);

/* fused gather + conv + bias; writes raw y and accumulates per-channel (sum, sumsq) of y in
 * bn_sums[2*Cout] (mg_sum, caller zeroes) for the following SpatialBatchNormalization */
int mg_conv_forward(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const void* wpack,
                    const float* bias, mg_grid* y, mg_sum* bn_sums);

/* nn.SpatialBatchNormalization statistics -> pending affine of the conv output.
 * training: batch stats from bn_sums over `count` elements per channel, running stats updated
 * (momentum, unbiased var); else running stats.  models/ilsvrc/rnmg.lua:27,37 */
int mg_bn_finalize(mg_ctx* ctx, const mg_sum* bn_sums, int64_t count, int32_t C, int32_t Cp,
                   const float* gamma, const float* beta, float* running_mean, float* running_var,
                   float eps, float momentum, int training,
                   float* scale, float* shift, float* save_mean, float* save_invstd);

/* out = relu?( T(z) + T(s)[c < s.C] ): CAddTable(true) + ReLU(true) with nn.Padding /
 * Identity shortcut (models/ilsvrc/rnmg.lua:13-20,140-154).  s may be NULL. */
int mg_residual_forward(mg_ctx* ctx, const mg_grid* z, const mg_grid* s, int relu, mg_grid* out, mg_grid* pooled);
/* `pooled` (nullable): also writes maxpool2x2_ceil(out) -- the operand the next stage's coarser
 * neighbour gathers (rnmg.lua:54-60), produced here so the conv's loader stays a pure copy */

/* mg_bn_finalize + mg_residual_forward as ONE pass: SpatialBatchNormalization (statistics -> affine, running
 * statistics update) -> [CAddTable(true) with the shortcut] -> [ReLU(true)] -> [pooled companion]
 * (models/ilsvrc/rnmg.lua:27,37 + 13-20,140-154).  z is the raw conv output; z->scale / z->shift must point at
 * [Cp] workspaces that receive the affine (kept for evaluation-time reuse and the fp32 path). */
typedef struct {
  const mg_sum* sums;   /* [2*C] (sum y, sum y^2) from mg_conv_forward / mg_bn_stats; unused when !training */
  int64_t count;        /* elements per channel behind the sums */
  const float* gamma;   /* nullable: 1 */
  const float* beta;    /* nullable: 0 */
  float* running_mean;  /* updated when training (nullable then); read when !training */
  float* running_var;
  float eps, momentum;
  int32_t training;
  float* save_mean;     /* nullable; [Cp] batch mean / invstd for mg_bn_backward */
  float* save_invstd;
} mg_bn_fused;
int mg_bn_residual_forward(mg_ctx* ctx, const mg_grid* z, const mg_bn_fused* bn, const mg_grid* s, int relu,
                           mg_grid* out, mg_grid* pooled);

/* per-channel (sum, sumsq) of a stored grid accumulated into bn_sums[2*C] (mg_sum, caller zeroes):
 * the statistics pass of nn.SpatialBatchNormalization when the conv epilogue did not fuse it */
int mg_bn_stats(mg_ctx* ctx, const mg_grid* y, mg_sum* bn_sums);
/* cudaMemsetAsync(ptr, 0, bytes) on the context stream (graph-capturable zeroing of sums/loss) */
int mg_memset_zero(mg_ctx* ctx, void* ptr, size_t bytes);

/* out[..., c_offset + c] = maxpool2x2_ceil(T(in))[..., c]  (mgPool, rnmg.lua:191-224);
 * argmax (nullable, int32 [N][Ho][Wo][C]) receives the flat y*W+x index, 0-based */
int mg_pool_forward(mg_ctx* ctx, const mg_grid* in, mg_grid* out, int32_t c_offset, int32_t* argmax);
/* out[..., c_offset + c] = T(in)[..., c]   (JoinTable(2) of mgPool isConcat) */
int mg_copy_channels(mg_ctx* ctx, const mg_grid* in, mg_grid* out, int32_t c_offset);
/* cudnn.SpatialAveragePooling(r,r,r,r) on NHWC (image pyramid, rnmg.lua:175-177) */
int mg_avgpool_forward(mg_ctx* ctx, const mg_grid* in, int32_t r, mg_grid* out);
/* im2col of the image-fed stem convolution cudnn.SpatialConvolution(3, C, 7,7, 2,2, 3,3) (rnmg.lua:180):
 * col[n][oy][ox][ci*k*k + ky*k + kx] = in[n][oy*stride-pad+ky][ox*stride-pad+kx][ci].  The channel order is Torch's
 * [Cout][Cin][kH][kW] weight layout flattened, so the stem becomes a 1x1 mg_conv over `col` that uses the module's
 * weight / gradWeight storage unchanged (K = 147 real channels instead of 49 taps x 8 padded ones).  bf16 only. */
int mg_im2col(mg_ctx* ctx, const mg_grid* in, int32_t ksize, int32_t stride, int32_t pad, mg_grid* col);
/* SpatialMaxPooling(3,3,2,2,1,1) of the ImageNet stem (rnmg.lua:183) */
int mg_pool3s2_forward(mg_ctx* ctx, const mg_grid* in, mg_grid* out, uint8_t* argmax_code /* nullable, bf16 mode */);
/* SpatialBatchNormalization -> ReLU -> SpatialMaxPooling(3,3,2,2,1,1) of the ImageNet stem (models/ilsvrc/rnmg.lua:181-183) as ONE pass
 * over the raw conv output z (bf16 contexts): BatchNorm finalisation as in mg_bn_residual_forward, pooled output + arg-max codes; the
 * full-resolution activation is never written.  Backward: mg_grad_combine with relu_mask = 2 (see there). */
int mg_bn_relu_pool3_forward(mg_ctx* ctx, const mg_grid* z, const mg_bn_fused* bn, mg_grid* out, uint8_t* argmax_code);
/* SelectTable(1) -> AvgPool(HxW) -> View: out[n][c] fp32 (rnmg.lua:281-283) */
int mg_global_avgpool_forward(mg_ctx* ctx, const mg_grid* in, mg_grid* out);
int mg_global_avgpool_backward(mg_ctx* ctx, const mg_grid* dout, mg_grid* din);

/* cudnn.SpatialFullConvolution(nIP, nOP, 2,2, 2,2, 0,0) -- the learned 2x up-sampling of U-MG
 * (models/mnist-cluttered/unmg.lua:35-52): y[n,2y+dy,2x+dx,co] = b[co] + sum_ci x[n,y,x,ci] * w[ci][co][dy][dx];
 * weight layout [nIP][nOP][2][2] as Torch stores it.  bn_sums as in mg_conv_forward.  backward: dx (nullable),
 * dw += gscale * ..., dbias += gscale * sum(g) (both nullable). */
int mg_upconv2x2_forward(mg_ctx* ctx, const mg_grid* x, const float* w, const float* bias, mg_grid* y, mg_sum* bn_sums);
int mg_upconv2x2_backward(mg_ctx* ctx, const mg_grid* x, const float* w, const mg_grid* g, mg_grid* dx,
                          float* dw, float* dbias, float gscale);

/* nn.Dropout(p) in training mode, Torch7's default (v2) form: y = x * mask * s, dx = dy * mask * s, mask in {0,1} with
 * P(keep) = 1 - p, s = fp32(1 / (1 - p)).  models/cifar/pnmg.lua:25-27 puts one in front of every convolution of blocks 2-5
 * when -isDropout.  The mask is counter based and never stored: element i, its NHWC index over the logical channels (pad
 * channels excluded), is kept iff word (i & 3) of Philox4x32-10(counter = (i >> 2, op, (uint32) *step, rank), key = (seed lo,
 * seed hi)) is >= t = min(2^32 - 1, floor(p * 2^32)).  *step is a device counter that mg_dropout_advance increments once per
 * training forward, so a captured CUDA graph draws a fresh mask on every replay; backward regenerates the forward's mask
 * from the same (seed, op, step, rank).  Every call rejects p < 0 and p >= 1. */
typedef struct {
  float p;               /* drop probability */
  uint32_t op;           /* ordinal of the dropout in the plan: masks of different dropouts are independent */
  uint32_t rank;         /* data-parallel rank (0 on one device): shards do not share masks */
  uint64_t seed;         /* Philox key */
  const uint64_t* step;  /* device */
} mg_dropout;
/* out = dropout(cat_C[ seg_0 | seg_1 | ... ]) as one tensor (pad channels written as zero).  seg_mode: MG_SEG_SAME (read at the
 * output resolution, pooled companions included) or MG_SEG_UP (coarser grid read at (y/2, x/2)); every mask element of an
 * up-sampled pixel is drawn independently, which is why the concatenation is materialised instead of gathered by the conv. */
int mg_dropout_forward(mg_ctx* ctx, const mg_dropout* dp, int32_t n_seg, const mg_grid* seg, const int32_t* seg_mode, mg_grid* out);
/* in place: g = g * mask * s (pad channels untouched) */
int mg_dropout_backward(mg_ctx* ctx, const mg_dropout* dp, mg_grid* g);
/* ++*step on the context stream */
int mg_dropout_advance(mg_ctx* ctx, uint64_t* step);

/* ---- backward ------------------------------------------------------------------------- */
/* Sum of all consumers' gradient contributions into tensor x (ConcatTable backward sums
 * its branches), routed through pool argmax / upsample block-sum, times the ReLU mask of x
 * when relu_mask.  Writes d (same shape as x).  If bn_sums != NULL also accumulates
 * (sum d, sum d*xraw) per channel with xraw = bn_x ? bn_x : x (raw data).
 * relu_mask = 2 (bf16): the tensor was never stored (mg_bn_relu_pool3_forward); x is its pooled form, the single source routes
 * through that call's arg-max codes and the mask of an element is the sign of the pooled value it was the arg-max of. */
int mg_grad_combine(mg_ctx* ctx, const mg_grid* x, int relu_mask, const mg_grid* bn_x,
                    int32_t n_src, const mg_grad_src* src, mg_grid* d, mg_sum* bn_sums);
/* BatchNorm backward given the sums: out = gamma*invstd*(d - mean(d) - xhat*mean(d*xhat))
 * (out may alias d); dgamma += gscale*sum(d*xhat); dbeta += gscale*sum(d).
 * conv_dbias (nullable): gradBias of the convolution that produced xraw, += gscale * sum_pixels(out),
 * fused here so that the weight-gradient call can be given dbias = NULL. */
int mg_bn_backward(mg_ctx* ctx, const mg_grid* xraw, const mg_grid* d, mg_grid* out, const mg_sum* bn_sums,
                   int64_t count, const float* gamma, const float* save_mean, const float* save_invstd,
                   float* dgamma, float* dbeta, float gscale, float* coef_ws /* [3*Cp] scratch */,
                   float* conv_dbias);
/* dcat = conv_transpose(g, w): gradient w.r.t. the concatenated input, segment s at channel
 * offset sum_{t<s} Cp_t */
int mg_conv_backward_data(mg_ctx* ctx, const mg_conv_desc* d, const float* w, const void* wpack_t,
                          const mg_grid* g, mg_grid* dcat);
/* dw += gscale * g^T * gather(x) ; dbias += gscale * sum(g)   (accGradParameters) */
int mg_conv_backward_weight(mg_ctx* ctx, const mg_conv_desc* d, const mg_grid* g,
                            float* dw, float* dbias, float gscale);

/* ---- one multigrid stage per call (plan level) ------------------------------------------
 * What a Torch7 host needs to stand in for the module graph mgConv() assembles (models/ilsvrc/rnmg.lua:91-159, residual;
 * models/cifar/nmg.lua:31-86, plain): tensors cross the boundary exactly as the reference's modules see them -- one NCHW fp32
 * device tensor per grid, finest first -- and parameters keep Torch's layout (conv weight [C_out][C_cat][k][k] with the input
 * planes ordered finer | same | coarser, bias [C_out]; BN weight / bias / running_mean / running_var [C_out]).  The plan holds
 * no device memory: mg_plan_workspace_bytes() tells the host how large a buffer (256-byte aligned, e.g. one CudaTensor) to
 * pass to every call; the same buffer must be passed to the backward call that follows a forward call.  The host need not
 * know anything about segments, pooled companions, epilogue fusion or gradient routing.
 * Index of the parameters of (layer l, grid i): l * n_scales + i; a residual unit has two layers, a plain stage one. */
enum { MG_STAGE_MAX_GRIDS = 4 };
typedef struct {
  int32_t n_scales;                       /* grids, finest first; H[i] == 2 * H[i+1] */
  int32_t C_in[MG_STAGE_MAX_GRIDS], C_out[MG_STAGE_MAX_GRIDS];
  int32_t H[MG_STAGE_MAX_GRIDS], W[MG_STAGE_MAX_GRIDS];
  int32_t ksize[MG_STAGE_MAX_GRIDS];      /* 3 (pad 1) or 1 (pad 0) per grid */
  int32_t residual;                       /* 1: ReLU(BN(mg(ReLU(BN(mg(x))))) + Shortcut(x)), Shortcut = Identity / nn.Padding (C_in <= C_out) */
  int32_t no_final_relu;                  /* isOut of models/mnist-cluttered/prnmg.mnist.lua:108-175 */
  float eps, momentum;                    /* of every SpatialBatchNormalization of the stage */
} mg_stage_desc;
typedef struct {
  const float* conv_w[2 * MG_STAGE_MAX_GRIDS]; const float* conv_b[2 * MG_STAGE_MAX_GRIDS];
  const float* bn_g[2 * MG_STAGE_MAX_GRIDS];   const float* bn_b[2 * MG_STAGE_MAX_GRIDS];
  float* bn_rm[2 * MG_STAGE_MAX_GRIDS];        float* bn_rv[2 * MG_STAGE_MAX_GRIDS];     /* running statistics, updated when training */
  float* conv_gw[2 * MG_STAGE_MAX_GRIDS];      float* conv_gb[2 * MG_STAGE_MAX_GRIDS];   /* gradWeight / gradBias: accumulated (+=) */
  float* bn_gg[2 * MG_STAGE_MAX_GRIDS];        float* bn_gb[2 * MG_STAGE_MAX_GRIDS];
} mg_stage_params;
typedef struct mg_stage_plan mg_stage_plan;
int mg_plan_create(mg_ctx* ctx, const mg_stage_desc* d, int32_t batch, mg_stage_plan** out);
size_t mg_plan_workspace_bytes(const mg_stage_plan* plan);
int mg_plan_destroy(mg_stage_plan* plan);
/* updateOutput: x[i] -> y[i] (NCHW fp32, [batch][C][H[i]][W[i]]); training != 0: batch statistics + running-statistics update */
int mg_stage_forward(mg_stage_plan* plan, void* workspace, const float* const* x, const mg_stage_params* params, float* const* y, int training);
/* updateGradInput + accGradParameters(scale): dy[i] -> dx[i] (dx or single entries may be NULL: no input gradient wanted) */
int mg_stage_backward(mg_stage_plan* plan, void* workspace, const float* const* dy, const mg_stage_params* params, float* const* dx, float scale);

/* ---- head / criterion / optimiser ("next" rows of the scope table) ------------------- */
/* LogSoftMax + ClassNLLCriterion (mean): logits grid N x 1 x 1 x C; target int32 0-based;
 * loss (1 float, device, caller zeroes) += NLL; logprob fp32 [N][C] (nullable);
 * dlogits = gscale * dloss/dlogits (nullable) */
int mg_nll_forward_backward(mg_ctx* ctx, const mg_grid* logits, const int32_t* target, float* logprob,
                            float* loss, mg_grid* dlogits, float gscale);
/* LogSoftMax alone (the model's last module, rnmg.lua:285) and its backward */
int mg_logsoftmax_forward(mg_ctx* ctx, const mg_grid* logits, float* logprob);
int mg_logsoftmax_backward(mg_ctx* ctx, const float* logprob, const float* grad_out, mg_grid* dlogits);
/* Sigmoid + BCECriterion (mean over elements) on a grid; target fp32 NCHW; loss += (caller zeroes) */
int mg_bce_forward_backward(mg_ctx* ctx, const mg_grid* x, const float* target_nchw, float* prob_nchw,
                            float* loss, mg_grid* dx, float gscale);
/* nn.Sigmoid alone: prob_nchw = sigmoid(T(x)); backward dx = grad_out * p * (1-p) */
int mg_sigmoid_forward(mg_ctx* ctx, const mg_grid* x, float* prob_nchw);
int mg_sigmoid_backward(mg_ctx* ctx, const float* prob_nchw, const float* grad_out_nchw, mg_grid* dx);
/* nn.ClassNLLCriterion (sizeAverage) on log-probabilities [N][C]: loss += -mean logprob[n][t[n]]
 * (caller zeroes); grad_out[N][C] (nullable) = -gscale/N at the target, 0 elsewhere */
int mg_nll_criterion(mg_ctx* ctx, const float* logprob, const int32_t* target, int32_t N, int32_t C,
                     float* loss, float* grad_out, float gscale);
/* nn.BCECriterion (sizeAverage, eps 1e-12) on probabilities, `count` elements */
int mg_bce_criterion(mg_ctx* ctx, const float* prob, const float* target, int64_t count,
                     float* loss, float* grad_prob, float gscale);
/* optim.sgd on a flat fp32 vector: g += wd*w; v = first ? g : mu*v+g; w -= lr*v */
int mg_sgd_step(mg_ctx* ctx, float* w, const float* g, float* v, int64_t n,
                float lr, float momentum, float wd, int first);

/* ---- data parallel (replaces nn.DataParallelTable, multigpu.lua:81-103) ---------------- */
int mg_comm_unique_id(void* out128);                                  /* ncclGetUniqueId */
int mg_comm_init(mg_ctx* ctx, int rank, int nranks, const void* id128);
int mg_comm_destroy(mg_ctx* ctx);
/* lend the communicator of `owner` (same device) to ctx: plans come and go with the input shape (the partial last
 * batch of pipelines/standard/test.lua:40-44 rebuilds them), the NCCL communicator must not.  ctx gets its own
 * communication stream; destroying ctx leaves the communicator alone, the owner must outlive every borrower. */
int mg_comm_share(mg_ctx* ctx, const mg_ctx* owner);
/* in-place sum all-reduce on the context's communication stream, ordered after everything
 * enqueued so far on the compute stream; mg_allreduce_wait makes the compute stream wait */
/* element type of the all-reduce calls: 0 = fp32, 1 = fp64, 2 = int64 (mg_sum buffers: 2 * n elements) */
int mg_allreduce_launch(mg_ctx* ctx, void* buf, int64_t count, int is_double);
int mg_allreduce_wait(mg_ctx* ctx);
/* in-place sum all-reduce enqueued on the COMPUTE stream itself: the cross-replica BatchNorm statistics
 * (sum, sumsq) forward and (sum d, sum d*y) backward of the -bnSync mode -- a few KB, latency bound */
int mg_allreduce_inline(mg_ctx* ctx, void* buf, int64_t count, int is_double);

#ifdef __cplusplus
}
#endif
#endif /* MGCONV_H */
