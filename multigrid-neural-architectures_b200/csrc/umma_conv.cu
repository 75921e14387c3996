// tcgen05 / TMEM implicit-GEMM multigrid convolution for sm_100a (bf16 operands, fp32 accumulate).
//
//   D[m][n] = sum_k A[m][k] * B[n][k]        m = output pixel (n, oy, ox), n = output channel
//
// K runs over "k-vectors" of 8 channels (16 bytes): for tap in k*k, for segment in the conv's
// gather list, for c8 in Cp_seg/8.  A is never materialised: four producer warps copy each
// k-vector of each of the CTA's 128 pixels straight from the source grids into the 128B-swizzled
// K-major operand image in shared memory with cp.async (zero-fill for the conv's zero padding);
// the same-scale grid, the pooled companion of the finer grid and the coarser grid (read at
// (y>>1, x>>1) -- SpatialUpSamplingNearest) are just different base pointers / shifts, so the
// channel concatenation of ResampleConcat (models/ilsvrc/rnmg.lua:41-89) exists only as the order
// of the K loop.  B (the weights) is pre-packed by pack_weights_kernel into exactly the shared
// memory image of each pipeline stage, so one thread moves a stage with a single cp.async.bulk.
// One elected thread issues tcgen05.mma (M=128, N<=256, K=16) into a TMEM accumulator; the
// producer warps drain it with tcgen05.ld, add the bias and store bf16 NHWC rows.
//
// forward:  A = gather(x),  B = W[co][(tap,ci)]                      -> y[m][co]
// dgrad  :  A = g (one SAME segment), B = W^T[cpad][(tap',co)], taps mirrored -> dcat[m][cpad]
// wgrad  :  see umma_wgrad.cu (MN-major operands).
#include "common.cuh"
#include "conv_view.cuh"
#include "umma_common.cuh"
#include "tma.cuh"
#include <algorithm>
#include <vector>

namespace {

constexpr int BM = 128;           // pixels per CTA = UMMA M
constexpr int KV_PER_STAGE = 8;   // 8 k-vectors of 8 bf16 = one 128-byte swizzle row
constexpr int A_STAGE_BYTES = BM * 128;
constexpr int N_PRODUCERS = 128;
constexpr int MMA_WARP = 4, B_WARP = 5;
constexpr int N_THREADS = 192;
constexpr int MAX_STAGES = 8;

struct UParams {
  USeg seg[MG_MAX_SEG];
  int n_seg;
  int k, stride, pad;
  int H, W;      // logical (concatenated) input size
  int Ho, Wo;
  int64_t M;     // N * Ho * Wo
  int Nimg;
  int kv_per_tap, nkv, n_stages;
  int n_tile;    // UMMA N of this launch (multiple of 16, <= 256)
  const uint8_t* wpack;  // [n_tiles][n_stages][n_tile][128B]
  const float* bias;     // [c_bias] or null
  int c_bias;
  __nv_bfloat16* y;
  int y_pitch;   // elements per output pixel
  int c_valid;   // channels to write (multiple of 8)
  int stages, lag;
  int tmem_cols;
  // halo kernel (3x3, stride 1): M rows are SLOTS of the zero-padded linear image space
  int Wp, Hp;        // slot pitch of an image row (W + 1) and rows per image (H + 1): the extra column / row is the conv's zero padding
  int64_t T;         // N * Hp * Wp slots
  int HL;            // halo slots staged per 64-channel chunk = 128 + 2 * Wp + 2
  int n_chunks;      // ceil(kv_per_tap / 8)
  int halo_bytes;    // HL * 128 rounded up to 1024
  int n_abuf;        // halo buffers (1 or 2)
  long long* timeline;   // debug (MGCONV_TIMELINE=1): per-CTA clock stamps [grid][8], else null
  mg_sum* stats;         // halo forward: per-channel (sum y, sum y^2) of the STORED bf16 output accumulated here ([2][c_stats]), or null
  int c_stats;
  // persistent halo kernel
  int m_tiles, n_ntiles, n_items;   // slot tiles, column tiles, work items = m_tiles * n_ntiles
};

// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, M=128
__host__ __device__ constexpr uint32_t idesc_bf16_m128(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// ---------------------------------------------------------------- the kernel ---------------
template <bool FAST>
__global__ void __launch_bounds__(N_THREADS, 4) umma_conv_kernel(const __grid_constant__ UParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // dynamic smem is only guaranteed 16-byte aligned: round up to the 1024 bytes the swizzle atoms need
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], tmem_full_bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ uint32_t s_row[BM];
  __shared__ USeg s_seg[MG_MAX_SEG];
  __shared__ float s_bias[256];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int S = p.stages;
  const int b_stage_bytes = p.n_tile * 128;
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + (size_t)S * A_STAGE_BYTES;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int ntile = blockIdx.y;

  if (tid < p.n_seg) s_seg[tid] = p.seg[tid];
  if (tid < BM) {  // packed (n, oy, ox) of this CTA's rows; 0xFFFFFFFF = row beyond M
    int64_t m = m0 + tid;
    uint32_t v = 0xFFFFFFFFu;
    if (m < p.M) {
      if (p.M < ((int64_t)1 << 32)) {   // 32-bit divisions: the prologue of 25 088 CTAs on the stem
        const uint32_t mu = (uint32_t)m, q = mu / (uint32_t)p.Wo, ox = mu - q * (uint32_t)p.Wo;
        const uint32_t n = q / (uint32_t)p.Ho, oy = q - n * (uint32_t)p.Ho;
        v = (n << 20) | (oy << 10) | ox;
      } else {
        int ox = (int)(m % p.Wo); int64_t q = m / p.Wo;
        int oy = (int)(q % p.Ho); int n = (int)(q / p.Ho);
        v = ((uint32_t)n << 20) | ((uint32_t)oy << 10) | (uint32_t)ox;
      }
    }
    s_row[tid] = v;
  }
  if (tid >= BM - 64 && tid < BM + 64) {   // bias tile of this column tile (zero beyond Cout): no global loads in the epilogue
    for (int c = tid - (BM - 64); c < p.n_tile; c += 128) {
      const int ch = blockIdx.y * p.n_tile + c;
      s_bias[c] = (p.bias && ch < p.c_bias) ? p.bias[ch] : 0.f;
    }
  }
  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(&full_bar[s], N_PRODUCERS + 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < 4) {
    // ================= A producers: gather k-vectors with cp.async ==========================
    const int v = tid & 7;       // k-vector slot of the stage (16-byte column of the 128-byte row)
    const int rg = tid >> 3;     // row group 0..15; rows rg, rg+16, ...
    const int L = p.lag;
    if (FAST) {
      // stride 1, "same" padding, k in {1,3}: everything that depends on the pixel is computed once per
      // CTA -- linear pixel index (SAME segments), half-resolution pixel index (UP segments) and a
      // validity bit per tap -- so that one k-vector copy costs a handful of instructions.
      uint32_t pix_up[BM / 16], flags[BM / 16];
      const uint32_t pix_same0 = (uint32_t)m0 + rg;   // pixel index of row it*16+rg = pix_same0 + it*16
      const int Hs2 = p.H >> 1, Ws2 = p.W >> 1;
#pragma unroll
      for (int it = 0; it < BM / 16; ++it) {
        const uint32_t ri = s_row[it * 16 + rg];
        const int ox = ri & 1023, oy = (ri >> 10) & 1023, n = ri >> 20;
        uint32_t f = 0;
        if (ri != 0xFFFFFFFFu) {
          for (int t = 0; t < p.k * p.k; ++t) {
            const int iy = oy + t / p.k - p.pad, ix = ox + t % p.k - p.pad;
            if ((unsigned)iy < (unsigned)p.H && (unsigned)ix < (unsigned)p.W) f |= 1u << t;
          }
          f |= (uint32_t)(oy & 1) << 9 | (uint32_t)(ox & 1) << 10;
          pix_up[it] = (uint32_t)(((size_t)n * Hs2 + (oy >> 1)) * Ws2 + (ox >> 1));
        } else {
          pix_up[it] = 0;
        }
        flags[it] = f;
      }
      const uint32_t dst_thread = (uint32_t)(rg * 128 + ((v ^ (rg & 7)) << 4));  // (it*16+rg)&7 == rg&7
      Ring rs(S), rpub(S);
      // this thread's k-vector j = ks * 8 + v as (tap = (ty, tx), r): carried along instead of three divisions per stage
      int tap = v / p.kv_per_tap, r = v - tap * p.kv_per_tap;
      int ty = tap / p.k, tx = tap - ty * p.k;
      for (int ks = 0; ks < p.n_stages + L; ++ks, rs.next()) {
        if (ks < p.n_stages) {
          const int s = rs.idx;
          if (ks >= S) mbar_wait(&empty_bar[s], rs.phase ^ 1u);
          const int j = ks * KV_PER_STAGE + v;
          const bool kv_ok = j < p.nkv;
          int sg = 0;
          if (kv_ok) while (sg + 1 < p.n_seg && r >= s_seg[sg + 1].kv_begin) ++sg;
          const USeg sgm = s_seg[sg];
          const int c8 = r - sgm.kv_begin;
          const int dy = ty - p.pad, dx = tx - p.pad;
          const uint32_t dst0 = smem_u32(a_smem + (size_t)s * A_STAGE_BYTES) + dst_thread;
          const uint32_t tapbit = kv_ok ? (1u << tap) : 0u;
          const uint32_t pitch = (uint32_t)sgm.Cp * 2u;
          const char* base = reinterpret_cast<const char*>(sgm.ptr) + c8 * 16;
          if (sgm.shift == 0) {
            base += (int64_t)(dy * p.W + dx) * (int64_t)pitch;
#pragma unroll
            for (int it = 0; it < BM / 16; ++it) {
              const bool ok = (flags[it] & tapbit) != 0;
              const char* src = ok ? base + (uint64_t)(pix_same0 + it * 16) * pitch : reinterpret_cast<const char*>(sgm.ptr);
              cp_async16(dst0 + it * 2048, src, ok ? 16u : 0u);
            }
          } else {
            // (o+d)>>1 - (o>>1):  d=-1 -> -1 if o even;  d=+1 -> +1 if o odd
#pragma unroll
            for (int it = 0; it < BM / 16; ++it) {
              const uint32_t f = flags[it];
              const bool ok = (f & tapbit) != 0;
              const int py = (f >> 9) & 1, px = (f >> 10) & 1;
              const int dyo = dy < 0 ? py - 1 : (dy > 0 ? py : 0);
              const int dxo = dx < 0 ? px - 1 : (dx > 0 ? px : 0);
              const char* src = ok ? base + (int64_t)((int64_t)pix_up[it] + dyo * Ws2 + dxo) * (int64_t)pitch
                                   : reinterpret_cast<const char*>(sgm.ptr);
              cp_async16(dst0 + it * 2048, src, ok ? 16u : 0u);
            }
          }
          r += KV_PER_STAGE;
          while (r >= p.kv_per_tap) { r -= p.kv_per_tap; ++tap; if (++tx == p.k) { tx = 0; ++ty; } }
        }
        cp_async_commit();
        if (ks >= L) {
          cp_async_wait_dyn(L);
          fence_proxy_async();
          mbar_arrive(&full_bar[rpub.idx]);
          rpub.next();
        }
      }
    } else {
      // general geometry (any k / stride / pad: the 7x7 stride-2 stem).  The kernel is issue bound (ncu: 59 % of the issue
      // slots on the stem), so everything that depends only on the row is decoded once per CTA: image index and the
      // input coordinates of tap (0,0); a copy then costs two adds, two bound checks and one address computation.
      int riy[BM / 16], rix[BM / 16], rn[BM / 16];
#pragma unroll
      for (int it = 0; it < BM / 16; ++it) {
        const uint32_t ri = s_row[it * 16 + rg];
        const bool valid = ri != 0xFFFFFFFFu;
        rn[it] = valid ? (int)(ri >> 20) : 0;
        riy[it] = valid ? (int)((ri >> 10) & 1023) * p.stride - p.pad : -(1 << 20);   // far outside: every bound check fails
        rix[it] = valid ? (int)(ri & 1023) * p.stride - p.pad : -(1 << 20);
      }
      const uint32_t dst_thread = (uint32_t)(rg * 128 + ((v ^ (rg & 7)) << 4));          // (it*16+rg)&7 == rg&7
      Ring rs(S), rpub(S);
      int tap = v / p.kv_per_tap, r = v - tap * p.kv_per_tap;
      int ty = tap / p.k, tx = tap - ty * p.k;
      for (int ks = 0; ks < p.n_stages + L; ++ks, rs.next()) {
        if (ks < p.n_stages) {
          const int s = rs.idx;
          if (ks >= S) mbar_wait(&empty_bar[s], rs.phase ^ 1u);
          // decode this lane's k-vector: (tap = (ty, tx), segment, channel offset), carried along from stage to stage
          const int j = ks * KV_PER_STAGE + v;
          const bool kv_ok = j < p.nkv;
          int sg = 0;
          if (kv_ok) while (sg + 1 < p.n_seg && r >= s_seg[sg + 1].kv_begin) ++sg;
          const USeg sgm = s_seg[sg];
          const int dy = kv_ok ? ty : -(1 << 20), dx = tx;
          const char* base = reinterpret_cast<const char*>(sgm.ptr) + (r - sgm.kv_begin) * 16;
          const uint32_t pitch = (uint32_t)sgm.Cp * 2u;
          const int plane = sgm.Hs * sgm.Ws;
          const uint32_t dst0 = smem_u32(a_smem + (size_t)s * A_STAGE_BYTES) + dst_thread;
#pragma unroll
          for (int it = 0; it < BM / 16; ++it) {
            const int iy = riy[it] + dy, ix = rix[it] + dx;
            const bool ok = (unsigned)iy < (unsigned)p.H && (unsigned)ix < (unsigned)p.W;
            const int64_t pixel = (int64_t)rn[it] * plane + (iy >> sgm.shift) * sgm.Ws + (ix >> sgm.shift);
            const char* src = ok ? base + pixel * pitch : reinterpret_cast<const char*>(sgm.ptr);
            cp_async16(dst0 + it * 2048, src, ok ? 16u : 0u);
          }
          r += KV_PER_STAGE;
          while (r >= p.kv_per_tap) { r -= p.kv_per_tap; if (++tx == p.k) { tx = 0; ++ty; } }
        }
        cp_async_commit();
        if (ks >= L) {  // stage ks-L has landed for this thread: publish it to the tensor core (async proxy)
          cp_async_wait_dyn(L);
          fence_proxy_async();
          mbar_arrive(&full_bar[rpub.idx]);
          rpub.next();
        }
      }
    }
    // ================= epilogue: TMEM -> registers -> bf16 NHWC rows ======================
    mbar_wait(&tmem_full_bar, 0);
    tc_fence_after();
    const int row = warp * 32 + lane;
    const int64_t m = m0 + row;
    const int n_base = ntile * p.n_tile;
    __nv_bfloat16* yrow = p.y + (size_t)(m < p.M ? m : 0) * p.y_pitch;
    for (int c0 = 0; c0 < p.n_tile; c0 += 16) {
      uint32_t acc[16];
      tc_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, acc);
      tc_wait_ld();
      if (m < p.M) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int n0 = n_base + c0 + h * 8;
          if (n0 + 8 <= p.c_valid) {
            uint32_t pk[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float a = __uint_as_float(acc[h * 8 + 2 * e]) + s_bias[c0 + h * 8 + 2 * e];
              const float b = __uint_as_float(acc[h * 8 + 2 * e + 1]) + s_bias[c0 + h * 8 + 2 * e + 1];
              __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
              pk[e] = *reinterpret_cast<uint32_t*>(&t);
            }
            *reinterpret_cast<uint4*>(yrow + n0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
      }
    }
    tc_fence_before();
  } else if (warp == B_WARP) {
    // ================= B loader: one bulk copy per stage =====================================
    if (lane == 0) {
      const uint8_t* wsrc = p.wpack + (size_t)ntile * p.n_stages * b_stage_bytes;
      Ring rs(S);
      for (int ks = 0; ks < p.n_stages; ++ks, rs.next()) {
        const int s = rs.idx;
        if (ks >= S) mbar_wait(&empty_bar[s], rs.phase ^ 1u);
        mbar_arrive_expect_tx(&full_bar[s], (uint32_t)b_stage_bytes);
        bulk_g2s(smem_u32(b_smem + (size_t)s * b_stage_bytes), wsrc + (size_t)ks * b_stage_bytes, (uint32_t)b_stage_bytes, &full_bar[s]);
      }
    }
  } else {
    // ================= MMA issuer: whole warp, elected lane issues (see elect_one) =================
    {
      const bool leader = elect_one();
      const uint32_t idesc = idesc_bf16_m128(p.n_tile);
      Ring rs(S);
      for (int ks = 0; ks < p.n_stages; ++ks, rs.next()) {
        const int s = rs.idx;
        mbar_wait(&full_bar[s], rs.phase);
        tc_fence_after();
        const uint32_t a_lo = desc_lo_k_sw128(smem_u32(a_smem + (size_t)s * A_STAGE_BYTES));
        const uint32_t b_lo = desc_lo_k_sw128(smem_u32(b_smem + (size_t)s * b_stage_bytes));
        const int kv_here = min(KV_PER_STAGE, p.nkv - ks * KV_PER_STAGE);
        const int ksteps = (kv_here + 1) >> 1;   // 16 bf16 = 2 k-vectors per UMMA K step
        if (leader) {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (q < ksteps) tc_mma_bf16_lohi(tmem_base, a_lo + q * 2, b_lo + q * 2, DESC_HI_SW128, idesc, (ks | q) != 0);
          tc_commit(&empty_bar[s]);   // frees the stage once these MMAs have read it
        }
      }
      if (leader) tc_commit(&tmem_full_bar);    // accumulator complete
    }
  }
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------- halo kernels ----------------
// 3x3 / stride 1 convolutions.  The CTA's 128 GEMM rows are 128 consecutive SLOTS of the zero-padded
// linear image space t = (n*(H+1) + y)*(W+1) + x (slot x == W and row y == H are the conv's zero
// padding, shared between neighbouring rows / images), so that tap (ky,kx) of every row is the slot
// (ky-1)*(W+1) + (kx-1) further on.  K is cut into CHUNKS of up to 64 channels of ONE source grid; per
// chunk the halo of the tile (128 + 2*(W+1) + 2 slots, widened to whole slot rows) is staged ONCE by
// the copy engine (TMA, tma.cuh): one cp.async.bulk.tensor per slot row, the zero padding and the
// nearest-neighbour up-sampling of the coarser grid included -- no thread touches an activation byte.
// The nine taps are nine UMMA descriptors into that same buffer, offset by whole 128-byte rows (the
// 128B swizzle is a function of the absolute shared-memory address, so a descriptor may start at any
// row -- scratch/desc_test.cu, scratch/tma_test.cu).  Weights stream as pre-swizzled stages
// (cp.async.bulk); a chunk of <= 32 (<= 16) channels packs 2 (4) taps into one 128-byte-row stage.

// butterfly reduce-scatter over the 32 lanes of a warp: every lane contributes v[0..15], afterwards lane l
// holds the warp-wide sum of element l & 15 (16 shuffles instead of 16 x 5)
__device__ __forceinline__ float warp_reduce_scatter16(float (&v)[16], int lane) {
#pragma unroll
  for (int o = 8; o >= 1; o >>= 1) {
    const bool hi = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = hi ? v[i] : v[i + o];
      const float keep = hi ? v[i + o] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}

constexpr int MAX_CHUNKS = 32;
struct HChunk { int seg, c0, nch, tps, ksteps, stage0; };   // tps = taps per weight stage (1, 2, 4); stage0 = first weight stage

struct HParams {
  CUtensorMap tmap[MG_MAX_SEG];
  int seg_up[MG_MAX_SEG];
  HChunk chunk[MAX_CHUNKS];
  int n_seg, n_chunks, n_stages, any_up;
  int img_box;        // whole-image TMA boxes (tma.cuh kind 4): the buffer is exactly the halo, (W+2) zero slots | tile | (W+2) zero slots
  int H, W, Wp, Hp, Nimg;
  int64_t T;          // N * Hp * Wp slots
  int HL;             // halo slots a tile needs = tile slots + 2 * Wp + 2
  int nr_max;         // slot rows a halo buffer holds
  int halo_bytes;     // nr_max * Wp * 128 rounded up to 1024
  int n_abuf;
  int n_tile;         // UMMA N of this launch (multiple of 16, <= 256)
  const uint8_t* wpack;
  const float* bias;
  int c_bias;
  __nv_bfloat16* y;
  int y_pitch, c_valid;
  int stages, tmem_cols;
  mg_sum* stats;      // forward: per-channel (sum y, sum y^2) of the STORED bf16 output accumulated here ([2][c_stats]), or null
  int c_stats;
  int m_tiles;        // persistent kernel: 128-slot tiles in total
  CUtensorMap tmap_w; // pair kernels: the packed weight image as rows of 128 bytes (tma.cuh kind 5)
  int tile_rows;      // persistent kernel, row-aligned tiles: a tile is tile_rows whole slot rows (tile_rows * Wp <= 128 slots), 0 = 128-slot tiles
  int epi_stage;      // halo / pair kernels: the epilogue stages every output row in shared memory (byte offset of the staging area + 1, 0 = direct
                      // stores) and hands it to the copy engine as ONE bulk store per row
};

// zero the pad column (slot x == W of every row) of `nbuf` halo buffers: the up-sampling box writes only the W valid slots
__device__ __forceinline__ void zero_pad_column(uint8_t* a_smem, int nbuf, int halo_bytes, int nr_max, int Wp, int tid, int nthreads, int org = 0) {
  for (int i = tid; i < nbuf * nr_max * 8; i += nthreads) {
    const int q = i & 7, row = (i >> 3) % nr_max, buf = (i >> 3) / nr_max;
    *reinterpret_cast<uint4*>(a_smem + (size_t)buf * halo_bytes + (size_t)(org + row * Wp + Wp - 1) * 128 + q * 16) = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async();
}

// whole-image mode: the Wp + 1 slots before and after the tile are never written by the copy engine; they are the zero pad row
// of the neighbouring image (before) and slots only padding outputs read (after) -- zero them once
__device__ __forceinline__ void zero_halo_margins(uint8_t* a_smem, int nbuf, int halo_bytes, int HL, int Wp, int tid, int nthreads) {
  const int m = Wp + 1;
  for (int i = tid; i < nbuf * 2 * m * 8; i += nthreads) {
    const int q = i & 7, sl = (i >> 3) % (2 * m), buf = (i >> 3) / (2 * m);
    const int slot = sl < m ? sl : HL - 2 * m + sl;
    *reinterpret_cast<uint4*>(a_smem + (size_t)buf * halo_bytes + (size_t)slot * 128 + q * 16) = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async();
}

// output pixel of slot t (or false for a padding slot / a slot beyond the batch)
__device__ __forceinline__ bool slot_pixel(const HParams& p, int64_t t, uint32_t* pix) {
  if (t >= p.T) return false;
  const uint32_t tu = (uint32_t)t, spi = (uint32_t)(p.Hp * p.Wp);
  const uint32_t n = tu / spi, rem = tu - n * spi;
  const uint32_t yy = rem / (uint32_t)p.Wp, xs = rem - yy * (uint32_t)p.Wp;
  if ((int)yy >= p.H || (int)xs >= p.W) return false;
  *pix = (n * p.H + yy) * p.W + xs;
  return true;
}

// MT = 128-slot sub-tiles per CTA (1 or 2).  With MT = 2 the CTA owns 256 consecutive slots and two TMEM accumulators:
// every weight stage feeds both sub-tiles, so the weight stream per output row halves and the halo overhead per row drops
// (the kernels are bound by L2 -> SM bandwidth, ~42 B/clk/SM chip-wide, of which the re-streamed weights are 70-90 %).
// Warps: 4*MT epilogue (TMEM lane quarters), one TMA warp for the halos, one thread for the weight stages, one MMA warp.
template <int MT>
__global__ void __launch_bounds__(32 * (4 * MT + 3), MT == 1 ? 4 : 2) umma_conv_halo_kernel(const __grid_constant__ HParams p) {
  constexpr int EPI_WARPS = 4 * MT, A_WARP = EPI_WARPS, B_WARP = EPI_WARPS + 1, M_WARP = EPI_WARPS + 2, NT = 32 * (EPI_WARPS + 3);
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], a_full[2], a_empty[2], tmem_full_bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_bias[256];                // bias of this column tile (zero beyond Cout): no global loads in the epilogue

  pdl_launch();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int S = p.stages;
  const int b_stage_bytes = p.n_tile * 128;
  uint8_t* a_smem = smem;                                      // halo buffers
  uint8_t* b_smem = smem + (size_t)p.n_abuf * p.halo_bytes;    // weight ring
  const int t0 = (int)blockIdx.x * (BM * MT);                  // T < 2^31 (halo_applies)
  const int ntile = blockIdx.y;
  // slot rows [r0, r0 + nr) cover the halo [hs, hs + HL); the tile's first halo slot sits `off` slots into the buffer
  const int hs = t0 - p.Wp - 1;
  const int r0 = floordiv(hs, p.Wp);
  const int nr = (hs + p.HL - 1) / p.Wp - r0 + 1;
  const int off = p.img_box ? 0 : hs - r0 * p.Wp;

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    mbar_init(&tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == M_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == A_WARP && lane < p.n_seg) tma_prefetch_desc(&p.tmap[lane]);
  if (p.img_box) zero_halo_margins(a_smem, p.n_abuf, p.halo_bytes, p.HL, p.Wp, tid, NT);
  else if (p.any_up) zero_pad_column(a_smem, p.n_abuf, p.halo_bytes, p.nr_max, p.Wp, tid, NT);
  // everything above touched only kernel parameters, shared memory and TMEM: it overlapped the tail of the
  // previous kernel; from here on the predecessor's output (activations, packed weights, bias) is read
  pdl_wait();
  for (int c = tid; c < p.n_tile; c += NT) {
    const int ch = blockIdx.y * p.n_tile + c;
    s_bias[c] = (p.bias && ch < p.c_bias) ? p.bias[ch] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < EPI_WARPS) {
    // ================= epilogue: TMEM -> registers -> bf16 NHWC rows ===========================
    // With p.stats the BatchNorm statistics of this tile (sum, sum of squares of the STORED bf16 values over the
    // valid rows) are reduced here: warp butterfly -> per-warp slots in the (now idle) halo buffer -> one deterministic
    // (fixed-point integer, mg_sum) atomic pair per channel and CTA.  The separate statistics pass over y (one HBM read of y) disappears.
    const int row = warp * 32 + lane;                      // sub-tile warp >> 2, TMEM lane quarter warp & 3
    uint32_t pix = 0;
    const bool row_ok = slot_pixel(p, (int64_t)t0 + row, &pix);
    const int n_base = ntile * p.n_tile;
    const bool want_stats = p.stats != nullptr;
    float* s_part = reinterpret_cast<float*>(a_smem);     // [4*MT warps][2][256]: every MMA has completed, the halo buffer is free
    __nv_bfloat16* yrow = p.y + (size_t)pix * p.y_pitch;
    const uint32_t tacc = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * p.n_tile);
    mbar_wait(&tmem_full_bar, 0);
    tc_fence_after();
    // Output rows leave through the copy engine: the lane writes its row (n_tile bf16 values) into a shared-memory staging row --
    // pitch n_tile * 2 + 16 bytes, so the 16-byte stores of a quarter warp hit distinct banks -- and issues ONE bulk store for it.
    // Direct stores are 2 * n_tile / 16 instructions per thread, each scattering 32 lanes over 32 different 128-byte lines: measured
    // (MG_PHASE_PROF) 9 300 cycles per 128 x 192 tile, a third of the CTA's lifetime.  Every MMA has completed: the halo buffers and
    // the weight ring are free.
    const int stage_pitch = p.n_tile * 2 + 16;
    uint8_t* stage_row = p.epi_stage ? smem + (p.epi_stage - 1) + (size_t)row * stage_pitch : nullptr;
    for (int c0 = 0; c0 < p.n_tile; c0 += 16) {
      uint32_t acc[16];
      tc_ld16(tacc + (uint32_t)c0, acc);
      tc_wait_ld();
      uint32_t pk[2][4];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int n0 = n_base + c0 + h * 8;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float a = __uint_as_float(acc[h * 8 + 2 * e]) + s_bias[c0 + h * 8 + 2 * e];
          const float b = __uint_as_float(acc[h * 8 + 2 * e + 1]) + s_bias[c0 + h * 8 + 2 * e + 1];
          __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
          pk[h][e] = *reinterpret_cast<uint32_t*>(&t);
        }
        if (stage_row) *reinterpret_cast<uint4*>(stage_row + (c0 + h * 8) * 2) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
        else if (row_ok && n0 + 8 <= p.c_valid) *reinterpret_cast<uint4*>(yrow + n0) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
      }
      if (want_stats) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const bool use = row_ok && n_base + c0 + h * 8 + 8 <= p.c_valid;
          float sv[16];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float ra = use ? __uint_as_float(pk[h][e] << 16) : 0.f, rb = use ? __uint_as_float(pk[h][e] & 0xFFFF0000u) : 0.f;
            sv[2 * e] = ra; sv[2 * e + 1] = rb;
            sv[8 + 2 * e] = ra * ra; sv[8 + 2 * e + 1] = rb * rb;
          }
          const float tot = warp_reduce_scatter16(sv, lane);   // lane l: (l & 15) < 8 -> sum of column, else sum of squares
          if (lane < 16) s_part[(warp * 2 + (lane >> 3)) * 256 + c0 + h * 8 + (lane & 7)] = tot;
        }
      }
    }
    if (stage_row) {
      const int ncols = min(p.n_tile, p.c_valid - n_base);          // columns of this tile inside the row pitch (multiple of 8)
      if (row_ok && ncols > 0) {
        fence_proxy_async();                                        // this thread's staging writes -> visible to the copy engine
        bulk_s2g(yrow + n_base, smem_u32(stage_row), (uint32_t)ncols * 2u);
        bulk_store_commit();
      }
    }
    tc_fence_before();
    if (want_stats) {
      asm volatile("bar.sync 1, %0;" ::"n"(128 * MT) : "memory");       // the epilogue warps
      for (int c = tid; c < p.n_tile; c += 128 * MT) {
        const int ch = n_base + c;
        if (ch < p.c_stats) {
          // every warp's sums (32 aligned slots, fixed butterfly order) enter as fixed-point integers: the totals do not depend
          // on how slots are grouped into CTAs, i.e. every kernel variant (TILE128 / TILE256 / RESIDENT) gives the same bits
          long long ah = 0, al = 0, bh = 0, bl = 0, h, l;
#pragma unroll
          for (int w = 0; w < 4 * MT; ++w) {
            mg_to_fix_f32(s_part[(2 * w) * 256 + c], h, l); ah += h; al += l;
            mg_to_fix_f32(s_part[(2 * w + 1) * 256 + c], h, l); bh += h; bl += l;
          }
          mg_sum_add_fix(p.stats + ch, ah, al);
          mg_sum_add_fix(p.stats + p.c_stats + ch, bh, bl);
        }
      }
    }
    if (stage_row) bulk_store_wait();   // the copy engine has read (and written) this thread's row before the CTA's shared memory goes away
  } else if (warp == A_WARP) {
    // ================= halo producer: one TMA per slot row and chunk ============================
    Ring ra(p.n_abuf);
    for (int c = 0; c < p.n_chunks; ++c, ra.next()) {
      const int buf = ra.idx;
      if (c >= p.n_abuf) mbar_wait(&a_empty[buf], ra.phase ^ 1u);
      const HChunk ch = p.chunk[c];
      const uint32_t dst = smem_u32(a_smem + (size_t)buf * p.halo_bytes);
      if (p.img_box) tma_load_images(&p.tmap[ch.seg], dst + (uint32_t)(p.Wp + 1) * 128u, &a_full[buf], ch.c0, t0 / (p.Hp * p.Wp), (uint32_t)(BM * MT) * 128u, lane);
      else tma_load_rows(&p.tmap[ch.seg], p.seg_up[ch.seg], dst, &a_full[buf], ch.c0, r0, nr, p.W, p.Hp, lane);
    }
  } else if (warp == B_WARP) {
    // ================= weight loader: one bulk copy per stage ====================================
    if (lane == 0) {
      const uint8_t* wsrc = p.wpack + (size_t)ntile * p.n_stages * b_stage_bytes;
      Ring rb(S);
      for (int ks = 0; ks < p.n_stages; ++ks, rb.next()) {
        const int s = rb.idx;
        if (ks >= S) mbar_wait(&empty_bar[s], rb.phase ^ 1u);
        mbar_arrive_expect_tx(&full_bar[s], (uint32_t)b_stage_bytes);
        bulk_g2s(smem_u32(b_smem + (size_t)s * b_stage_bytes), wsrc + (size_t)ks * b_stage_bytes, (uint32_t)b_stage_bytes, &full_bar[s]);
      }
    }
  } else {
    // ================= MMA issuer: 9 shifted descriptors per chunk ===============================
    // the whole warp runs the loop (warp-uniform operands), the elected lane issues the MMAs and the commits
    const bool leader = elect_one();
    const uint32_t idesc = idesc_bf16_m128(p.n_tile);
    Ring ra(p.n_abuf), rb(S);
    for (int c = 0; c < p.n_chunks; ++c, ra.next()) {
      const int buf = ra.idx;
      const HChunk ch = p.chunk[c];
      mbar_wait(&a_full[buf], ra.phase);
      tc_fence_after();
      const uint32_t a_base = smem_u32(a_smem + (size_t)buf * p.halo_bytes) + (uint32_t)off * 128u;
      const int tps = ch.tps, ksteps = ch.ksteps;
      const uint32_t sub_lo = 8u / (uint32_t)tps;          // descriptor units (16 bytes) between the taps packed in one stage
      int sub = 0;
      uint32_t b_lo = 0;
      for (int tap = 0; tap < 9; ++tap) {
        if (sub == 0) {
          mbar_wait(&full_bar[rb.idx], rb.phase);
          tc_fence_after();
          b_lo = desc_lo_k_sw128(smem_u32(b_smem + (size_t)rb.idx * b_stage_bytes));
        }
        const uint32_t a_lo = desc_lo_k_sw128(a_base + (uint32_t)((tap / 3) * p.Wp + (tap % 3)) * 128u);
        const bool last_of_stage = (sub == tps - 1) || tap == 8;
        if (leader) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)   // both sub-tiles consume the same weight stage
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (q < ksteps) {
                tc_mma_bf16_lohi(tmem_base + (uint32_t)(mt * p.n_tile), a_lo + (uint32_t)(mt * BM * 8 + q * 2), b_lo + (uint32_t)sub * sub_lo + (uint32_t)(q * 2),
                                 DESC_HI_SW128, idesc, (uint32_t)((c | tap | q) != 0));
              }
          if (last_of_stage) tc_commit(&empty_bar[rb.idx]);   // frees the weight stage once these MMAs have read it
        }
        if (last_of_stage) { sub = 0; rb.next(); } else ++sub;
      }
      if (leader) tc_commit(&a_empty[buf]);   // halo buffer free once this chunk's MMAs have read it
    }
    if (leader) tc_commit(&tmem_full_bar);
  }
  __syncthreads();
  if (warp == M_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------- CTA-pair halo kernel ----------
// The same operand scheme on tcgen05 CTA pairs (cta_group::2): the two CTAs of a cluster own two consecutive tiles; ONE MMA
// instruction (M = 256) issued by the even CTA drives the tensor cores of both SMs, each reading its own halo (A) and HALF of the
// weight stage (N / 2 rows of B) from its own shared memory.  Per SM the weight stream -- what bounds the N >= 128 layers at the
// chip's L2 -> SM rate -- halves, and the ring holds twice the stages in the same memory.  Every copy of either CTA counts its
// bytes on the EVEN CTA's barriers (cp.async.bulk.tensor.cta_group::2); tcgen05.commit multicasts the "stage free" / "accumulator
// complete" arrivals to both CTAs.  The tile's first halo slot sits Wp slots into the buffer in BOTH CTAs (the MMA's A descriptor
// is one address for the pair), so each CTA lands its rows Wp - off slots in.
template <int MT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(32 * (4 * MT + 3), MT == 1 ? 4 : 2) umma_conv_halo_pair_kernel(const __grid_constant__ HParams p) {
  constexpr int EPI_WARPS = 4 * MT, A_WARP = EPI_WARPS, B_WARP = EPI_WARPS + 1, M_WARP = EPI_WARPS + 2, NT = 32 * (EPI_WARPS + 3);
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], a_full[2], a_empty[2], tmem_full_bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_bias[256];

  pdl_launch();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int S = p.stages;
  const int b_half_bytes = (p.n_tile >> 1) * 128;              // this CTA's half of a weight stage
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + (size_t)p.n_abuf * p.halo_bytes;
  const int t0 = (int)blockIdx.x * (BM * MT);
  const int ntile = blockIdx.y;
  const int hs = t0 - p.Wp - 1;
  const int r0 = floordiv(hs, p.Wp);
  const int nr = (hs + p.HL - 1) / p.Wp - r0 + 1;
  const int off = hs - r0 * p.Wp;
  const int org = p.img_box ? 0 : p.Wp - off;                  // slots: where this CTA's first slot row lands in the buffer
  const int a_first = p.img_box ? 0 : p.Wp;                    // slots: the tile's first halo slot, the same in both CTAs

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    mbar_init(&tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == M_WARP) {   // the same warp of both CTAs allocates the pair's columns
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (warp == A_WARP && lane < p.n_seg) tma_prefetch_desc(&p.tmap[lane]);
  if (warp == B_WARP && lane == 0) tma_prefetch_desc(&p.tmap_w);
  if (p.img_box) zero_halo_margins(a_smem, p.n_abuf, p.halo_bytes, p.HL, p.Wp, tid, NT);
  else if (p.any_up) zero_pad_column(a_smem, p.n_abuf, p.halo_bytes, p.nr_max, p.Wp, tid, NT, org);
  pdl_wait();
  for (int c = tid; c < p.n_tile; c += NT) {
    const int ch = blockIdx.y * p.n_tile + c;
    s_bias[c] = (p.bias && ch < p.c_bias) ? p.bias[ch] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // both CTAs' barriers are initialised before any remote completion can arrive
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < EPI_WARPS) {
    // ================= epilogue (per CTA: its own 128 * MT rows x all N columns) =================
    const int row = warp * 32 + lane;
    uint32_t pix = 0;
    const bool row_ok = slot_pixel(p, (int64_t)t0 + row, &pix);
    const int n_base = ntile * p.n_tile;
    const bool want_stats = p.stats != nullptr;
    float* s_part = reinterpret_cast<float*>(a_smem);
    __nv_bfloat16* yrow = p.y + (size_t)pix * p.y_pitch;
    const uint32_t tacc = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * p.n_tile);
    mbar_wait_cluster(&tmem_full_bar, 0);
    tc_fence_after();
    // Output rows leave through the copy engine: the lane writes its row (n_tile bf16 values) into a shared-memory staging row --
    // pitch n_tile * 2 + 16 bytes, so the 16-byte stores of a quarter warp hit distinct banks -- and issues ONE bulk store for it.
    // Direct stores are 2 * n_tile / 16 instructions per thread, each scattering 32 lanes over 32 different 128-byte lines: measured
    // (MG_PHASE_PROF) 9 300 cycles per 128 x 192 tile, a third of the CTA's lifetime.  Every MMA has completed: the halo buffers and
    // the weight ring are free.
    const int stage_pitch = p.n_tile * 2 + 16;
    uint8_t* stage_row = p.epi_stage ? smem + (p.epi_stage - 1) + (size_t)row * stage_pitch : nullptr;
    for (int c0 = 0; c0 < p.n_tile; c0 += 16) {
      uint32_t acc[16];
      tc_ld16(tacc + (uint32_t)c0, acc);
      tc_wait_ld();
      uint32_t pk[2][4];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int n0 = n_base + c0 + h * 8;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float a = __uint_as_float(acc[h * 8 + 2 * e]) + s_bias[c0 + h * 8 + 2 * e];
          const float b = __uint_as_float(acc[h * 8 + 2 * e + 1]) + s_bias[c0 + h * 8 + 2 * e + 1];
          __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
          pk[h][e] = *reinterpret_cast<uint32_t*>(&t);
        }
        if (stage_row) *reinterpret_cast<uint4*>(stage_row + (c0 + h * 8) * 2) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
        else if (row_ok && n0 + 8 <= p.c_valid) *reinterpret_cast<uint4*>(yrow + n0) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
      }
      if (want_stats) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const bool use = row_ok && n_base + c0 + h * 8 + 8 <= p.c_valid;
          float sv[16];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float ra = use ? __uint_as_float(pk[h][e] << 16) : 0.f, rb = use ? __uint_as_float(pk[h][e] & 0xFFFF0000u) : 0.f;
            sv[2 * e] = ra; sv[2 * e + 1] = rb;
            sv[8 + 2 * e] = ra * ra; sv[8 + 2 * e + 1] = rb * rb;
          }
          const float tot = warp_reduce_scatter16(sv, lane);
          if (lane < 16) s_part[(warp * 2 + (lane >> 3)) * 256 + c0 + h * 8 + (lane & 7)] = tot;
        }
      }
    }
    if (stage_row) {
      const int ncols = min(p.n_tile, p.c_valid - n_base);          // columns of this tile inside the row pitch (multiple of 8)
      if (row_ok && ncols > 0) {
        fence_proxy_async();                                        // this thread's staging writes -> visible to the copy engine
        bulk_s2g(yrow + n_base, smem_u32(stage_row), (uint32_t)ncols * 2u);
        bulk_store_commit();
      }
    }
    tc_fence_before();
    if (want_stats) {
      asm volatile("bar.sync 1, %0;" ::"n"(128 * MT) : "memory");
      for (int c = tid; c < p.n_tile; c += 128 * MT) {
        const int ch = n_base + c;
        if (ch < p.c_stats) {
          long long ah = 0, al = 0, bh = 0, bl = 0, h, l;
#pragma unroll
          for (int w = 0; w < 4 * MT; ++w) {
            mg_to_fix_f32(s_part[(2 * w) * 256 + c], h, l); ah += h; al += l;
            mg_to_fix_f32(s_part[(2 * w + 1) * 256 + c], h, l); bh += h; bl += l;
          }
          mg_sum_add_fix(p.stats + ch, ah, al);
          mg_sum_add_fix(p.stats + p.c_stats + ch, bh, bl);
        }
      }
    }
    if (stage_row) bulk_store_wait();   // the copy engine has read (and written) this thread's row before the CTA's shared memory goes away
  } else if (warp == A_WARP) {
    // ================= halo producer: this CTA's rows, bytes counted on the even CTA's barrier =================
    // bytes the pair lands per chunk: rows of both tiles (the even CTA knows its peer's geometry)
    const int hs_p = t0 + BM * MT - p.Wp - 1;
    const int r0_p = floordiv(hs_p, p.Wp);
    const int nr_p = (hs_p + p.HL - 1) / p.Wp - r0_p + 1;
    Ring ra(p.n_abuf);
    for (int c = 0; c < p.n_chunks; ++c, ra.next()) {
      const int buf = ra.idx;
      if (c >= p.n_abuf) mbar_wait_cluster(&a_empty[buf], ra.phase ^ 1u);
      const HChunk ch = p.chunk[c];
      const uint32_t dst = smem_u32(a_smem + (size_t)buf * p.halo_bytes);
      if (p.img_box) {
        if (lane == 0) {
          if (rank == 0) mbar_arrive_expect_tx(&a_full[buf], 2u * (uint32_t)(BM * MT) * 128u);
          tma_load_4d_pair(dst + (uint32_t)(p.Wp + 1) * 128u, &p.tmap[ch.seg], &a_full[buf], ch.c0, 0, 0, t0 / (p.Hp * p.Wp));
        }
      } else {
        const int up = p.seg_up[ch.seg];
        if (rank == 0 && lane == 0) mbar_arrive_expect_tx(&a_full[buf], (uint32_t)(nr + nr_p) * (uint32_t)(up ? p.W : p.Wp) * 128u);
        __syncwarp();
        tma_load_rows_pair(&p.tmap[ch.seg], up, dst + (uint32_t)org * 128u, &a_full[buf], ch.c0, r0, nr, p.W, p.Hp, lane);
      }
    }
  } else if (warp == B_WARP) {
    // ================= weight loader: this CTA's half of every stage =================
    if (lane == 0) {
      const int row0 = ntile * p.n_stages * p.n_tile + (int)rank * (p.n_tile >> 1);
      Ring rb(S);
      for (int ks = 0; ks < p.n_stages; ++ks, rb.next()) {
        const int s = rb.idx;
        if (ks >= S) mbar_wait_cluster(&empty_bar[s], rb.phase ^ 1u);
        if (rank == 0) mbar_arrive_expect_tx(&full_bar[s], 2u * (uint32_t)b_half_bytes);
        tma_load_2d_pair(smem_u32(b_smem + (size_t)s * b_half_bytes), &p.tmap_w, &full_bar[s], 0, row0 + ks * p.n_tile);
      }
    }
  } else if (rank == 0) {
    // ================= MMA issuer (even CTA only): M = 256 across the pair =================
    const bool leader = elect_one();
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    Ring ra(p.n_abuf), rb(S);
    for (int c = 0; c < p.n_chunks; ++c, ra.next()) {
      const int buf = ra.idx;
      const HChunk ch = p.chunk[c];
      mbar_wait_cluster(&a_full[buf], ra.phase);
      tc_fence_after();
      const uint32_t a_base = smem_u32(a_smem + (size_t)buf * p.halo_bytes) + (uint32_t)a_first * 128u;
      const int tps = ch.tps, ksteps = ch.ksteps;
      const uint32_t sub_lo = 8u / (uint32_t)tps;
      int sub = 0;
      uint32_t b_lo = 0;
      for (int tap = 0; tap < 9; ++tap) {
        if (sub == 0) {
          mbar_wait_cluster(&full_bar[rb.idx], rb.phase);
          tc_fence_after();
          b_lo = desc_lo_k_sw128(smem_u32(b_smem + (size_t)rb.idx * b_half_bytes));
        }
        const uint32_t a_lo = desc_lo_k_sw128(a_base + (uint32_t)((tap / 3) * p.Wp + (tap % 3)) * 128u);
        const bool last_of_stage = (sub == tps - 1) || tap == 8;
        if (leader) {
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (q < ksteps) {
                tc_mma_bf16_lohi_pair(tmem_base + (uint32_t)(mt * p.n_tile), a_lo + (uint32_t)(mt * BM * 8 + q * 2), b_lo + (uint32_t)sub * sub_lo + (uint32_t)(q * 2),
                                      DESC_HI_SW128, idesc, (uint32_t)((c | tap | q) != 0));
              }
          if (last_of_stage) tc_commit_pair(&empty_bar[rb.idx]);
        }
        if (last_of_stage) { sub = 0; rb.next(); } else ++sub;
      }
      if (leader) tc_commit_pair(&a_empty[buf]);
    }
    if (leader) tc_commit_pair(&tmem_full_bar);
  }
  __syncthreads();
  cluster_sync_all();     // neither CTA leaves (or frees TMEM) while its peer may still read its shared memory or signal its barriers
  if (warp == M_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------- persistent halo kernel ----------
// Same operand scheme for convolutions whose WHOLE packed weight image fits in shared memory next to a ring of halo
// buffers (R-MG-34 block 1: 96 -> 64 at 56x56 is 112 KB, its dgrad 110 KB).  The non-persistent kernel re-streams the
// weights for every 128-slot tile -- 2.4x the activation traffic at N = 64.  Here one CTA per SM loads the weights ONCE,
// then walks slot tiles blockIdx.x, +gridDim.x, ... with decoupled roles:
//   1 TMA warp       stages halos into a ring that runs ACROSS chunks and tiles (the next tile's halo is in flight while
//                    the tensor core works on the current one),
//   1 MMA warp       accumulates tile i into TMEM accumulator i & 1 (every operand already in shared memory),
//   4 epilogue warps drain accumulator (i-1) & 1 meanwhile (TMEM double buffering) and keep the BatchNorm
//                    statistics of all the CTA's tiles in shared memory: one deterministic (integer) atomic pair per channel and CTA.
constexpr int P_A_WARP = 8, P_B_WARP = 9, P_MMA_WARP = 10, P_THREADS = 352;   // 2 x 4 epilogue warps (one group per TMEM accumulator), TMA, weights, MMA
constexpr int P_MAX_ABUF = 6;

__global__ void __launch_bounds__(P_THREADS, 1) umma_conv_halo_persistent_kernel(const __grid_constant__ HParams p) {
  pdl_launch();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t b_full, a_full[P_MAX_ABUF], a_empty[P_MAX_ABUF], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NA = p.n_abuf;
  const int b_stage_bytes = p.n_tile * 128;
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + (size_t)NA * p.halo_bytes;                                  // all weight stages, resident
  long long* s_part = reinterpret_cast<long long*>(b_smem + (size_t)p.n_stages * b_stage_bytes);   // [4 epilogue warps][2][n_tile][hi, lo]
  float* s_bias = reinterpret_cast<float*>(s_part + 32 * p.n_tile);                    // [n_tile]
  const int n_my = (p.m_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles blockIdx.x, +gridDim.x, ...
  // Row-aligned tiles (tile_rows > 0): a tile is R whole slot rows, its halo exactly the R + 2 rows around it plus one slot on either
  // side.  The slot before (the pad slot of row r - 2: always zero) is buffer slot 0, zeroed once; rows land from buffer slot 1.
  // Against 128-slot tiles at arbitrary offsets (halo = up to 6 rows of a 56-wide grid for 2.25 rows of outputs) the halo buffer
  // shrinks by a third, which is what lets the ring run a tile ahead of the tensor core next to the resident weights.
  const int R = p.tile_rows;
  const int tile_slots = R ? R * p.Wp : BM;

  for (int c = tid; c < 32 * p.n_tile; c += P_THREADS) s_part[c] = 0;
  if (tid == 0) {
    mbar_init(&b_full, 1);
    for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == P_MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == P_A_WARP && lane < p.n_seg) tma_prefetch_desc(&p.tmap[lane]);
  if (p.img_box) zero_halo_margins(a_smem, NA, p.halo_bytes, p.HL, p.Wp, tid, P_THREADS);
  else if (p.any_up) zero_pad_column(a_smem, NA, p.halo_bytes, p.nr_max, p.Wp, tid, P_THREADS, R ? 1 : 0);
  if (R) {   // buffer slot 0 and the slot after the last row: never written by the copy engine
    for (int i = tid; i < NA * 2 * 8; i += P_THREADS) {
      const int q = i & 7, which = (i >> 3) & 1, buf = i >> 4;
      const int slot = which ? 1 + (R + 2) * p.Wp : 0;
      *reinterpret_cast<uint4*>(a_smem + (size_t)buf * p.halo_bytes + (size_t)slot * 128 + q * 16) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
  }
  pdl_wait();
  for (int c = tid; c < p.n_tile; c += P_THREADS) s_bias[c] = (p.bias && c < p.c_bias) ? p.bias[c] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < 8) {
    // ================= epilogue: warps 0-3 drain accumulator 0 (even tiles), warps 4-7 accumulator 1 (odd tiles) ==========
    // (with the BatchNorm sums one group of four warps needs ~4 600 cycles per 64-column tile, the MMAs ~3 300: measured with
    // MG_PHASE_PROF; two groups keep the drain off the critical path)
    const int grp = warp >> 2, qw = warp & 3;
    const bool want_stats = p.stats != nullptr;
#ifdef MG_PHASE_PROF
    long long e_wait = 0, e_work = 0;
#endif
    for (int it = grp; it < n_my; it += 2) {
      const int mt = blockIdx.x + it * gridDim.x;
      const int acc = it & 1;
      const int row = qw * 32 + lane;
      uint32_t pix = 0;
      const bool row_ok = row < tile_slots && slot_pixel(p, (int64_t)mt * tile_slots + row, &pix);
#ifdef MG_PHASE_PROF
      const long long e0 = clock64();
#endif
      mbar_wait(&tmem_full[acc], (it >> 1) & 1);
      tc_fence_after();
#ifdef MG_PHASE_PROF
      const long long e1 = clock64();
#endif
      __nv_bfloat16* yrow = p.y + (size_t)pix * p.y_pitch;
      const uint32_t tcol = tmem_base + ((uint32_t)(qw * 32) << 16) + (uint32_t)(acc * p.n_tile);
      for (int c0 = 0; c0 < p.n_tile; c0 += 16) {
        uint32_t a16[16];
        tc_ld16(tcol + (uint32_t)c0, a16);
        tc_wait_ld();
        uint32_t pk[2][4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int n0 = c0 + h * 8;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float a = __uint_as_float(a16[h * 8 + 2 * e]) + s_bias[c0 + h * 8 + 2 * e];
            const float b = __uint_as_float(a16[h * 8 + 2 * e + 1]) + s_bias[c0 + h * 8 + 2 * e + 1];
            __nv_bfloat162 t2 = __floats2bfloat162_rn(a, b);
            pk[h][e] = *reinterpret_cast<uint32_t*>(&t2);
          }
          if (row_ok && n0 + 8 <= p.c_valid) *reinterpret_cast<uint4*>(yrow + n0) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
        }
        if (want_stats) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const bool use = row_ok && c0 + h * 8 + 8 <= p.c_valid;
            float sv[16];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float ra = use ? __uint_as_float(pk[h][e] << 16) : 0.f, rb = use ? __uint_as_float(pk[h][e] & 0xFFFF0000u) : 0.f;
              sv[2 * e] = ra; sv[2 * e + 1] = rb;
              sv[8 + 2 * e] = ra * ra; sv[8 + 2 * e + 1] = rb * rb;
            }
            const float tot = warp_reduce_scatter16(sv, lane);
            // slot owned by this lane of this warp for the whole kernel: accumulate over the CTA's tiles without synchronisation,
            // as fixed-point integers (exact, so the totals do not depend on which tiles this CTA happened to walk)
            if (lane < 16) {
              long long fh, fl;
              mg_to_fix_f32(tot, fh, fl);
              long long* sp = s_part + (size_t)((warp * 2 + (lane >> 3)) * p.n_tile + c0 + h * 8 + (lane & 7)) * 2;
              sp[0] += fh; sp[1] += fl;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);   // 128 arrivals: the accumulator may be overwritten
#ifdef MG_PHASE_PROF
      e_wait += e1 - e0; e_work += clock64() - e1;
#endif
    }
#ifdef MG_PHASE_PROF
    if (blockIdx.x == 3 && tid == 0) printf("epilogue warp0: tiles %d wait_tmem_full %lld work %lld cycles/tile\n", n_my, e_wait / n_my, e_work / n_my);
#endif
    if (want_stats) {
      asm volatile("bar.sync 3, 256;" ::: "memory");
      for (int c = tid; c < p.n_tile; c += 256)
        if (c < p.c_stats) {
          long long ah = 0, al = 0, bh = 0, bl = 0;
#pragma unroll
          for (int w = 0; w < 8; ++w) {
            const long long* sa = s_part + (size_t)((w * 2) * p.n_tile + c) * 2;
            const long long* sb = s_part + (size_t)((w * 2 + 1) * p.n_tile + c) * 2;
            ah += sa[0]; al += sa[1]; bh += sb[0]; bl += sb[1];
          }
          mg_sum_add_fix(p.stats + c, ah, al);
          mg_sum_add_fix(p.stats + p.c_stats + c, bh, bl);
        }
    }
  } else if (warp == P_A_WARP) {
    // ================= halo producer: the ring runs across chunks and tiles =======================
    Ring ra(NA);
    int ac = 0;
    for (int it = 0; it < n_my; ++it) {
      const int t0 = (int)(blockIdx.x + it * gridDim.x) * tile_slots;
      const int hs = t0 - p.Wp - 1;
      const int r0 = R ? t0 / p.Wp - 1 : floordiv(hs, p.Wp);
      const int nr = R ? R + 2 : (hs + p.HL - 1) / p.Wp - r0 + 1;
      for (int c = 0; c < p.n_chunks; ++c, ++ac, ra.next()) {
        const int buf = ra.idx;
        if (ac >= NA) mbar_wait(&a_empty[buf], ra.phase ^ 1u);
        const HChunk ch = p.chunk[c];
        const uint32_t dst = smem_u32(a_smem + (size_t)buf * p.halo_bytes) + (R ? 128u : 0u);
        if (p.img_box) tma_load_images(&p.tmap[ch.seg], dst + (uint32_t)(p.Wp + 1) * 128u, &a_full[buf], ch.c0, t0 / (p.Hp * p.Wp), (uint32_t)BM * 128u, lane);
        else tma_load_rows(&p.tmap[ch.seg], p.seg_up[ch.seg], dst, &a_full[buf], ch.c0, r0, nr, p.W, p.Hp, lane);
      }
    }
  } else if (warp == P_B_WARP) {
    // ================= weight loader: every stage once =============================================
    if (lane == 0) {
      mbar_arrive_expect_tx(&b_full, (uint32_t)(p.n_stages * b_stage_bytes));
      for (int q = 0; q < p.n_stages; ++q)
        bulk_g2s(smem_u32(b_smem + (size_t)q * b_stage_bytes), p.wpack + (size_t)q * b_stage_bytes, (uint32_t)b_stage_bytes, &b_full);
    }
  } else {
    // ================= MMA issuer (whole warp, elected lane issues; see elect_one) =================
    const bool leader = elect_one();
    const uint32_t idesc = idesc_bf16_m128(p.n_tile);
    const uint32_t b_base = smem_u32(b_smem);
    Ring ra(NA);
    mbar_wait(&b_full, 0);
#ifdef MG_PHASE_PROF
    long long m_wait_e = 0, m_wait_a = 0, m_issue = 0, m_t0 = clock64();
#endif
    for (int it = 0; it < n_my; ++it) {
      const int acc = it & 1;
#ifdef MG_PHASE_PROF
      const long long q0 = clock64();
#endif
      if (it >= 2) { mbar_wait(&tmem_empty[acc], ((it >> 1) - 1) & 1); tc_fence_after(); }
#ifdef MG_PHASE_PROF
      m_wait_e += clock64() - q0;
#endif
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.n_tile);
      const int t0 = (int)(blockIdx.x + it * gridDim.x) * tile_slots;
      const int hs = t0 - p.Wp - 1;
      const int off = (p.img_box || R) ? 0 : hs - floordiv(hs, p.Wp) * p.Wp;
      for (int c = 0; c < p.n_chunks; ++c, ra.next()) {
        const int buf = ra.idx;
        const HChunk ch = p.chunk[c];
#ifdef MG_PHASE_PROF
        const long long q1 = clock64();
#endif
        mbar_wait(&a_full[buf], ra.phase);
        tc_fence_after();
#ifdef MG_PHASE_PROF
        const long long q2 = clock64();
        m_wait_a += q2 - q1;
#endif
        const uint32_t a_base = smem_u32(a_smem + (size_t)buf * p.halo_bytes) + (uint32_t)off * 128u;
        const int tps = ch.tps, ksteps = ch.ksteps;
        const uint32_t sub_lo = 8u / (uint32_t)tps;
        if (leader) {
          int sub = 0, st = ch.stage0;
          for (int tap = 0; tap < 9; ++tap) {
            const uint32_t a_lo = desc_lo_k_sw128(a_base + (uint32_t)((tap / 3) * p.Wp + (tap % 3)) * 128u);
            const uint32_t b_lo = desc_lo_k_sw128(b_base + (uint32_t)(st * b_stage_bytes)) + (uint32_t)sub * sub_lo;
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (q < ksteps) tc_mma_bf16_lohi(d_tmem, a_lo + (uint32_t)(q * 2), b_lo + (uint32_t)(q * 2), DESC_HI_SW128, idesc, (uint32_t)((c | tap | q) != 0));
            if (++sub == tps) { sub = 0; ++st; }
          }
          tc_commit(&a_empty[buf]);
        }
#ifdef MG_PHASE_PROF
        m_issue += clock64() - q2;
#endif
      }
      if (leader) tc_commit(&tmem_full[acc]);
    }
#ifdef MG_PHASE_PROF
    if (blockIdx.x == 3 && lane == 0) printf("MMA warp: tiles %d total %lld wait_tmem_empty %lld wait_a_full %lld issue %lld cycles/tile\n", n_my, (clock64() - m_t0) / n_my, m_wait_e / n_my, m_wait_a / n_my, m_issue / n_my);
#endif
  }
  __syncthreads();
  if (warp == P_MMA_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------- persistent CTA-pair halo kernel ----------
// The weight-resident kernel on tcgen05 CTA pairs: each CTA keeps HALF of every weight stage (so the ring of halos next to it is
// deep enough to run two tiles ahead: on the 56 x 56 layers the single-CTA kernel holds 115 KB of weights and two halo buffers, and
// every tile exposes the copy engine's latency), the pair walks tile pairs (2 * (pair + it * P) + rank), one M = 256 MMA per K step
// serves both tiles.  Needs a tile offset that is the same in both CTAs: row-aligned tiles or whole-image boxes.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(P_THREADS, 1) umma_conv_halo_persistent_pair_kernel(const __grid_constant__ HParams p) {
  pdl_launch();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t b_full, a_full[P_MAX_ABUF], a_empty[P_MAX_ABUF], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int NA = p.n_abuf;
  const int b_half_bytes = (p.n_tile >> 1) * 128;
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + (size_t)NA * p.halo_bytes;                                  // this CTA's half of all weight stages
  long long* s_part = reinterpret_cast<long long*>(b_smem + (size_t)p.n_stages * b_half_bytes);
  float* s_bias = reinterpret_cast<float*>(s_part + 32 * p.n_tile);
  const int R = p.tile_rows;
  const int tile_slots = R ? R * p.Wp : BM;
  const int pair = (int)blockIdx.x >> 1, P = (int)gridDim.x >> 1;
  const int pair_tiles = (p.m_tiles + 1) >> 1;                                         // tile pairs in total
  const int n_my = (pair_tiles - pair + P - 1) / P;                                    // the same in both CTAs of a pair

  for (int c = tid; c < 32 * p.n_tile; c += P_THREADS) s_part[c] = 0;
  if (tid == 0) {
    mbar_init(&b_full, 1);
    for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 256); }   // epilogue threads of both CTAs
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == P_MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (warp == P_A_WARP && lane < p.n_seg) tma_prefetch_desc(&p.tmap[lane]);
  if (warp == P_B_WARP && lane == 0) tma_prefetch_desc(&p.tmap_w);
  if (p.img_box) zero_halo_margins(a_smem, NA, p.halo_bytes, p.HL, p.Wp, tid, P_THREADS);
  else if (p.any_up) zero_pad_column(a_smem, NA, p.halo_bytes, p.nr_max, p.Wp, tid, P_THREADS, R ? 1 : 0);
  if (R) {
    for (int i = tid; i < NA * 2 * 8; i += P_THREADS) {
      const int q = i & 7, which = (i >> 3) & 1, buf = i >> 4;
      const int slot = which ? 1 + (R + 2) * p.Wp : 0;
      *reinterpret_cast<uint4*>(a_smem + (size_t)buf * p.halo_bytes + (size_t)slot * 128 + q * 16) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
  }
  pdl_wait();
  for (int c = tid; c < p.n_tile; c += P_THREADS) s_bias[c] = (p.bias && c < p.c_bias) ? p.bias[c] : 0.f;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < 8) {
    // ================= epilogue: this CTA's tile of the pair; warps 0-3 even iterations, warps 4-7 odd ones ===========
    const int grp = warp >> 2, qw = warp & 3;
    const bool want_stats = p.stats != nullptr;
    for (int it = grp; it < n_my; it += 2) {
      const int mt = 2 * (pair + it * P) + (int)rank;
      const int acc = it & 1;
      const int row = qw * 32 + lane;
      uint32_t pix = 0;
      const bool row_ok = mt < p.m_tiles && row < tile_slots && slot_pixel(p, (int64_t)mt * tile_slots + row, &pix);
      mbar_wait_cluster(&tmem_full[acc], (it >> 1) & 1);
      tc_fence_after();
      __nv_bfloat16* yrow = p.y + (size_t)pix * p.y_pitch;
      const uint32_t tcol = tmem_base + ((uint32_t)(qw * 32) << 16) + (uint32_t)(acc * p.n_tile);
      for (int c0 = 0; c0 < p.n_tile; c0 += 16) {
        uint32_t a16[16];
        tc_ld16(tcol + (uint32_t)c0, a16);
        tc_wait_ld();
        uint32_t pk[2][4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int n0 = c0 + h * 8;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float a = __uint_as_float(a16[h * 8 + 2 * e]) + s_bias[c0 + h * 8 + 2 * e];
            const float b = __uint_as_float(a16[h * 8 + 2 * e + 1]) + s_bias[c0 + h * 8 + 2 * e + 1];
            __nv_bfloat162 t2 = __floats2bfloat162_rn(a, b);
            pk[h][e] = *reinterpret_cast<uint32_t*>(&t2);
          }
          if (row_ok && n0 + 8 <= p.c_valid) *reinterpret_cast<uint4*>(yrow + n0) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
        }
        if (want_stats) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const bool use = row_ok && c0 + h * 8 + 8 <= p.c_valid;
            float sv[16];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float ra = use ? __uint_as_float(pk[h][e] << 16) : 0.f, rb = use ? __uint_as_float(pk[h][e] & 0xFFFF0000u) : 0.f;
              sv[2 * e] = ra; sv[2 * e + 1] = rb;
              sv[8 + 2 * e] = ra * ra; sv[8 + 2 * e + 1] = rb * rb;
            }
            const float tot = warp_reduce_scatter16(sv, lane);
            if (lane < 16) {
              long long fh, fl;
              mg_to_fix_f32(tot, fh, fl);
              long long* sp = s_part + (size_t)((warp * 2 + (lane >> 3)) * p.n_tile + c0 + h * 8 + (lane & 7)) * 2;
              sp[0] += fh; sp[1] += fl;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive_cluster(&tmem_empty[acc], 0);   // 256 arrivals on the even CTA's barrier: both tiles drained
    }
    if (want_stats) {
      asm volatile("bar.sync 3, 256;" ::: "memory");
      for (int c = tid; c < p.n_tile; c += 256)
        if (c < p.c_stats) {
          long long ah = 0, al = 0, bh = 0, bl = 0;
#pragma unroll
          for (int w = 0; w < 8; ++w) {
            const long long* sa = s_part + (size_t)((w * 2) * p.n_tile + c) * 2;
            const long long* sb = s_part + (size_t)((w * 2 + 1) * p.n_tile + c) * 2;
            ah += sa[0]; al += sa[1]; bh += sb[0]; bl += sb[1];
          }
          mg_sum_add_fix(p.stats + c, ah, al);
          mg_sum_add_fix(p.stats + p.c_stats + c, bh, bl);
        }
    }
  } else if (warp == P_A_WARP) {
    // ================= halo producer: this CTA's tile; bytes of both CTAs counted on the even CTA's barrier ==========
    Ring ra(NA);
    int ac = 0;
    for (int it = 0; it < n_my; ++it) {
      const int t0 = (2 * (pair + it * P) + (int)rank) * tile_slots;
      const int r0 = t0 / p.Wp - 1;
      const int nr = R + 2;
      for (int c = 0; c < p.n_chunks; ++c, ++ac, ra.next()) {
        const int buf = ra.idx;
        if (ac >= NA) mbar_wait_cluster(&a_empty[buf], ra.phase ^ 1u);
        const HChunk ch = p.chunk[c];
        const uint32_t dst = smem_u32(a_smem + (size_t)buf * p.halo_bytes) + (R ? 128u : 0u);
        if (p.img_box) {
          if (lane == 0) {
            if (rank == 0) mbar_arrive_expect_tx(&a_full[buf], 2u * (uint32_t)BM * 128u);
            tma_load_4d_pair(dst + (uint32_t)(p.Wp + 1) * 128u, &p.tmap[ch.seg], &a_full[buf], ch.c0, 0, 0, t0 / (p.Hp * p.Wp));
          }
        } else {
          const int up = p.seg_up[ch.seg];
          if (rank == 0 && lane == 0) mbar_arrive_expect_tx(&a_full[buf], 2u * (uint32_t)nr * (uint32_t)(up ? p.W : p.Wp) * 128u);
          __syncwarp();
          tma_load_rows_pair(&p.tmap[ch.seg], up, dst, &a_full[buf], ch.c0, r0, nr, p.W, p.Hp, lane);
        }
      }
    }
  } else if (warp == P_B_WARP) {
    // ================= weight loader: this CTA's half of every stage, once =============================
    if (lane == 0) {
      if (rank == 0) mbar_arrive_expect_tx(&b_full, (uint32_t)(2 * p.n_stages * b_half_bytes));
      for (int q = 0; q < p.n_stages; ++q)
        tma_load_2d_pair(smem_u32(b_smem + (size_t)q * b_half_bytes), &p.tmap_w, &b_full, 0, q * p.n_tile + (int)rank * (p.n_tile >> 1));
    }
  } else if (rank == 0) {
    // ================= MMA issuer (even CTA): M = 256 across the pair =================
    const bool leader = elect_one();
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    const uint32_t b_base = smem_u32(b_smem);
    Ring ra(NA);
    mbar_wait_cluster(&b_full, 0);
    for (int it = 0; it < n_my; ++it) {
      const int acc = it & 1;
      if (it >= 2) { mbar_wait_cluster(&tmem_empty[acc], ((it >> 1) - 1) & 1); tc_fence_after(); }
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.n_tile);
      for (int c = 0; c < p.n_chunks; ++c, ra.next()) {
        const int buf = ra.idx;
        const HChunk ch = p.chunk[c];
        mbar_wait_cluster(&a_full[buf], ra.phase);
        tc_fence_after();
        const uint32_t a_base = smem_u32(a_smem + (size_t)buf * p.halo_bytes);
        const int tps = ch.tps, ksteps = ch.ksteps;
        const uint32_t sub_lo = 8u / (uint32_t)tps;
        if (leader) {
          int sub = 0, st = ch.stage0;
          for (int tap = 0; tap < 9; ++tap) {
            const uint32_t a_lo = desc_lo_k_sw128(a_base + (uint32_t)((tap / 3) * p.Wp + (tap % 3)) * 128u);
            const uint32_t b_lo = desc_lo_k_sw128(b_base + (uint32_t)(st * b_half_bytes)) + (uint32_t)sub * sub_lo;
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (q < ksteps) tc_mma_bf16_lohi_pair(d_tmem, a_lo + (uint32_t)(q * 2), b_lo + (uint32_t)(q * 2), DESC_HI_SW128, idesc, (uint32_t)((c | tap | q) != 0));
            if (++sub == tps) { sub = 0; ++st; }
          }
          tc_commit_pair(&a_empty[buf]);
        }
      }
      if (leader) tc_commit_pair(&tmem_full[acc]);
    }
  }
  __syncthreads();
  cluster_sync_all();
  if (warp == P_MMA_WARP) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}


// ---------------------------------------------------------------- stem kernel ----------------
// cudnn.SpatialConvolution(3, C, 7,7, 2,2, 3,3) on the image pyramid (models/ilsvrc/rnmg.lua:180): 2.3 % of the MACs of R-MG-34
// but, as an im2col gather of 49 taps x 16 bytes per output pixel, 0.8 ms of the step on the generic kernel.  Here nothing is
// gathered at all.  A tile is 16 x 8 output pixels; the copy engine loads its input patch (37 rows x 21 pixels x 8 channels,
// out-of-bounds = the conv's zero padding) and four warps split it into two PARITY PLANES (even / odd input columns),
// 37 rows x 11 pixels each.  (Loading the planes directly with elementStrides = 2 works -- first version of this kernel -- but
// the copy engine then fetches 16 bytes per request and becomes the bottleneck: 2 600 cycles per tile against 900 of MMAs.)  In a plane the 8 output pixels of a tile row read, for a given tap column, 8 CONSECUTIVE 16-byte pixels
// -- exactly one UMMA core matrix (8 rows x 16 bytes) of a K-major no-swizzle operand -- and the next tile row is two plane rows
// further (SBO); taps kx = 2q and 2q+1 sit at the same offset of the even and the odd plane (LBO).  So im2col is 28 shared-
// memory descriptors per tile (7 kernel rows x 4 column pairs, K = 16 = two taps x 8 channels), and the tensor core reads the
// patch in place.  Weights (7 stages of [Cout][64 K]) stay resident; the CTA is persistent over tiles with a ring of patches
// and two TMEM accumulators; the epilogue (bias, bf16 store, BatchNorm sums) is the persistent halo kernel's.
constexpr int ST_PC = 11, ST_PR = 37;                    // plane columns / rows
constexpr int ST_ROW = ST_PC * 16;                       // 176 bytes per plane row
constexpr int ST_PLANE = 6592;                           // plane stride (>= 37 * 176 = 6512; = 64 mod 128: the two K halves of an MMA row group sit in different banks)
constexpr int ST_SLOT = 13312;                           // two planes, multiple of 256
constexpr int ST_MAX_RING = 6;
constexpr int ST_RAW_COLS = 21;                          // input columns of a tile's patch (2 * 8 + 5)
constexpr int ST_RAW = 12544;                            // raw patch 37 x 21 x 16 bytes = 12432, rounded up to 128
constexpr int ST_THREADS = 480;                          // 2 x 4 epilogue warps (one group per TMEM accumulator), TMA, weights, MMA, 4 de-interleave warps

struct StemParams {
  CUtensorMap tmap;          // kind 2 map of the input image grid (Cp = 8): patch boxes
  CUtensorMap tmap_y;        // kind 3 map of the output grid (TMA store of 16 x 8 x 64-channel tiles), used when tma_out
  int tma_out;               // n_tile == 64 == y pitch: the epilogue stages the tile in shared memory and the copy engine stores it
  int H, W, Ho, Wo, Nimg;
  int tiles_x, tiles_y, n_tiles_total;
  int n_tile;                // UMMA N (Cout rounded up to 16)
  int ring;
  const uint8_t* wpack;      // [7][n_tile][128 B]
  const float* bias; int c_bias;
  __nv_bfloat16* y; int y_pitch, c_valid;
  mg_sum* stats; int c_stats;
  int tmem_cols;
};

__device__ __forceinline__ uint64_t smem_desc_k_none(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}

__global__ void __launch_bounds__(ST_THREADS, 1) umma_stem_kernel(const __grid_constant__ StemParams p) {
  pdl_launch();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t b_full, r_full[ST_MAX_RING], r_empty[ST_MAX_RING], a_full[ST_MAX_RING], a_empty[ST_MAX_RING], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NA = p.ring;
  const int b_stage_bytes = p.n_tile * 128;
  uint8_t* b_smem = smem;                                           // 7 weight stages, resident
  uint8_t* a_smem = smem + 7 * b_stage_bytes;                       // ring of plane pairs (what the tensor core reads)
  uint8_t* r_smem = a_smem + (size_t)NA * ST_SLOT;                  // ring of raw patches (what the copy engine writes)
  uint8_t* o_smem = r_smem + (size_t)NA * ST_RAW;                   // two output staging tiles (128 rows x 128 bytes, swizzled), when tma_out
  long long* s_part = reinterpret_cast<long long*>(o_smem + (p.tma_out ? 2 * 16384 : 0));   // [8 warps][2][n_tile][hi, lo]
  float* s_bias = reinterpret_cast<float*>(s_part + 32 * p.n_tile);
  const int n_my = (p.n_tiles_total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  for (int c = tid; c < 32 * p.n_tile; c += ST_THREADS) s_part[c] = 0;
  if (tid == 0) {
    mbar_init(&b_full, 1);
    for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 128); mbar_init(&a_empty[s], 1); mbar_init(&r_full[s], 1); mbar_init(&r_empty[s], 128); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 10) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == 8 && lane == 0) tma_prefetch_desc(&p.tmap);
  // column 10 of every odd plane belongs to the non-existent tap kx = 7 (zero weights): it is never written, so it must hold
  // finite values -- zero it once
  for (int i = tid; i < NA * ST_PR; i += ST_THREADS) {
    const int sl = i / ST_PR, r = i - sl * ST_PR;
    *reinterpret_cast<uint4*>(a_smem + (size_t)sl * ST_SLOT + ST_PLANE + r * ST_ROW + 10 * 16) = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async();
  pdl_wait();
  for (int c = tid; c < p.n_tile; c += ST_THREADS) s_bias[c] = (p.bias && c < p.c_bias) ? p.bias[c] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  const int tiles_per_img = p.tiles_x * p.tiles_y;

  if (warp < 8) {
    // ================= epilogue: warps 0-3 drain accumulator 0 (even tiles), warps 4-7 accumulator 1 (odd tiles) =================
    // (the tile's MMAs take ~900 cycles; one group of four warps needs longer than that for TMEM -> bf16 rows + BatchNorm sums)
    const bool want_stats = p.stats != nullptr;
    const int grp = warp >> 2, qw = warp & 3;
    uint8_t* stage = o_smem + grp * 16384;
    for (int it = grp; it < n_my; it += 2) {
      const int tile = blockIdx.x + it * gridDim.x;
      const int n = tile / tiles_per_img, tr = tile - n * tiles_per_img;
      const int ty = tr / p.tiles_x, tx = tr - ty * p.tiles_x;
      const int acc = it & 1;
      const int row = qw * 32 + lane;                      // TMEM lane = tile row (row >> 3), tile column (row & 7)
      const int oy = ty * 16 + (row >> 3), ox = tx * 8 + (row & 7);
      const bool row_ok = oy < p.Ho && ox < p.Wo;
      mbar_wait(&tmem_full[acc], (it >> 1) & 1);
      tc_fence_after();
      if (p.tma_out) {   // the previous tile's store has read the staging buffer
        if (qw == 0 && lane == 0) tma_store_wait_read();
        if (grp == 0) asm volatile("bar.sync 4, 128;" ::: "memory"); else asm volatile("bar.sync 5, 128;" ::: "memory");
      }
      __nv_bfloat16* yrow = p.y + ((size_t)((size_t)n * p.Ho + (row_ok ? oy : 0)) * p.Wo + (row_ok ? ox : 0)) * p.y_pitch;
      const uint32_t tcol = tmem_base + ((uint32_t)(qw * 32) << 16) + (uint32_t)(acc * p.n_tile);
      // two TMEM loads in flight per wait (the loop is latency bound: load -> wait -> convert -> store)
      for (int c00 = 0; c00 < p.n_tile; c00 += 32) {
        uint32_t a32[2][16];
        const bool two = c00 + 16 < p.n_tile;
        tc_ld16(tcol + (uint32_t)c00, a32[0]);
        if (two) tc_ld16(tcol + (uint32_t)(c00 + 16), a32[1]);
        tc_wait_ld();
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (u == 1 && !two) break;
          const int c0 = c00 + u * 16;
          uint32_t pk[2][4];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int n0 = c0 + h * 8;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float a = __uint_as_float(a32[u][h * 8 + 2 * e]) + s_bias[c0 + h * 8 + 2 * e];
              const float b = __uint_as_float(a32[u][h * 8 + 2 * e + 1]) + s_bias[c0 + h * 8 + 2 * e + 1];
              __nv_bfloat162 t2 = __floats2bfloat162_rn(a, b);
              pk[h][e] = *reinterpret_cast<uint32_t*>(&t2);
            }
            if (p.tma_out) {   // 16-byte chunk n0 / 8 of row `row`, 128-byte swizzle: conflict-free, un-swizzled by the TMA store
              *reinterpret_cast<uint4*>(stage + row * 128 + ((((n0 >> 3) ^ (row & 7))) << 4)) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
            } else if (row_ok && n0 + 8 <= p.c_valid) {
              *reinterpret_cast<uint4*>(yrow + n0) = make_uint4(pk[h][0], pk[h][1], pk[h][2], pk[h][3]);
            }
          }
          if (want_stats) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const bool use = row_ok && c0 + h * 8 + 8 <= p.c_valid;
              float sv[16];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float ra = use ? __uint_as_float(pk[h][e] << 16) : 0.f, rb = use ? __uint_as_float(pk[h][e] & 0xFFFF0000u) : 0.f;
                sv[2 * e] = ra; sv[2 * e + 1] = rb;
                sv[8 + 2 * e] = ra * ra; sv[8 + 2 * e + 1] = rb * rb;
              }
              const float tot = warp_reduce_scatter16(sv, lane);
              if (lane < 16) {
                long long fh, fl;
                mg_to_fix_f32(tot, fh, fl);
                long long* sp = s_part + (size_t)((warp * 2 + (lane >> 3)) * p.n_tile + c0 + h * 8 + (lane & 7)) * 2;
                sp[0] += fh; sp[1] += fl;
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
      if (p.tma_out) {   // tile staged: hand it to the copy engine (rows / columns beyond the image are clipped by the tensor map)
        fence_proxy_async();
        if (grp == 0) asm volatile("bar.sync 4, 128;" ::: "memory"); else asm volatile("bar.sync 5, 128;" ::: "memory");
        if (qw == 0 && lane == 0) {
          tma_store_4d(&p.tmap_y, smem_u32(stage), 0, tx * 8, ty * 16, n);
          tma_store_commit();
        }
      }
    }
    if (p.tma_out && qw == 0 && lane == 0) tma_store_wait_all();
    if (want_stats) {
      asm volatile("bar.sync 3, 256;" ::: "memory");
      for (int c = tid; c < p.n_tile; c += 256)
        if (c < p.c_stats) {
          long long ah = 0, al = 0, bh = 0, bl = 0;
#pragma unroll
          for (int w = 0; w < 8; ++w) {
            const long long* sa = s_part + (size_t)((w * 2) * p.n_tile + c) * 2;
            const long long* sb = s_part + (size_t)((w * 2 + 1) * p.n_tile + c) * 2;
            ah += sa[0]; al += sa[1]; bh += sb[0]; bl += sb[1];
          }
          mg_sum_add_fix(p.stats + c, ah, al);
          mg_sum_add_fix(p.stats + p.c_stats + c, bh, bl);
        }
    }
  } else if (warp == 8) {
    // ================= patch producer: one box of 37 rows x 21 pixels per tile =================
    if (lane == 0) {
      Ring rr(NA);
      for (int it = 0; it < n_my; ++it, rr.next()) {
        const int tile = blockIdx.x + it * gridDim.x;
        const int n = tile / tiles_per_img, tr = tile - n * tiles_per_img;
        const int ty = tr / p.tiles_x, tx = tr - ty * p.tiles_x;
        const int s = rr.idx;
        if (it >= NA) mbar_wait(&r_empty[s], rr.phase ^ 1u);
        mbar_arrive_expect_tx(&r_full[s], (uint32_t)(ST_PR * ST_RAW_COLS * 16));
        tma_load_4d(smem_u32(r_smem + (size_t)s * ST_RAW), &p.tmap, &r_full[s], 0, 2 * tx * 8 - 3, 2 * ty * 16 - 3, n);
      }
    }
  } else if (warp >= 11) {
    // ================= de-interleave: raw patch -> even / odd column planes =================
    const int dt = tid - 11 * 32;
    Ring rr(NA);
    for (int it = 0; it < n_my; ++it, rr.next()) {
      const int s = rr.idx;
      mbar_wait(&r_full[s], rr.phase);
      if (it >= NA) mbar_wait(&a_empty[s], rr.phase ^ 1u);      // the MMAs that read this plane slot have completed
      const uint8_t* raw = r_smem + (size_t)s * ST_RAW;
      uint8_t* pl = a_smem + (size_t)s * ST_SLOT;
      for (int i = dt; i < ST_PR * ST_RAW_COLS; i += 128) {
        const int r = i / ST_RAW_COLS, x = i - r * ST_RAW_COLS;
        const uint4 v = *reinterpret_cast<const uint4*>(raw + (size_t)i * 16);
        *reinterpret_cast<uint4*>(pl + (x & 1) * ST_PLANE + r * ST_ROW + (x >> 1) * 16) = v;
      }
      fence_proxy_async();              // generic-proxy writes -> visible to the tensor core (async proxy)
      mbar_arrive(&a_full[s]);
      mbar_arrive(&r_empty[s]);
    }
  } else if (warp == 9) {
    if (lane == 0) {
      mbar_arrive_expect_tx(&b_full, (uint32_t)(7 * b_stage_bytes));
      for (int q = 0; q < 7; ++q) bulk_g2s(smem_u32(b_smem + (size_t)q * b_stage_bytes), p.wpack + (size_t)q * b_stage_bytes, (uint32_t)b_stage_bytes, &b_full);
    }
  } else {
    // ================= MMA issuer: 7 kernel rows x 4 column pairs per tile =================
    const bool leader = elect_one();
    const uint32_t idesc = idesc_bf16_m128(p.n_tile);
    const uint32_t b_base = smem_u32(b_smem);
    Ring ra(NA);
    mbar_wait(&b_full, 0);
    for (int it = 0; it < n_my; ++it, ra.next()) {
      const int acc = it & 1;
      if (it >= 2) { mbar_wait(&tmem_empty[acc], ((it >> 1) - 1) & 1); tc_fence_after(); }
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.n_tile);
      const int s = ra.idx;
      mbar_wait(&a_full[s], ra.phase);
      tc_fence_after();
      const uint32_t a_base = smem_u32(a_smem + (size_t)s * ST_SLOT);
      if (leader) {
#pragma unroll 1
        for (int ky = 0; ky < 7; ++ky) {
          const uint64_t b_desc = smem_desc_k_sw128(b_base + (uint32_t)(ky * b_stage_bytes));
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint64_t a_desc = smem_desc_k_none(a_base + (uint32_t)(ky * ST_ROW + q * 16), ST_PLANE, 2 * ST_ROW);
            tc_mma_bf16(d_tmem, a_desc, b_desc + (uint64_t)(q * 2), idesc, (uint32_t)((ky | q) != 0));
          }
        }
        tc_commit(&a_empty[s]);
        tc_commit(&tmem_full[acc]);
      }
    }
  }
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

// ---------------------------------------------------------------- weight packing -----------
struct PackParams {
  const float* w;   // [Cout][Ccat][k][k]
  uint8_t* out;
  int transposed;
  int k, Ccat, Cout;
  int n_seg;
  int seg_C[MG_MAX_SEG], seg_cbegin[MG_MAX_SEG], seg_kvbegin[MG_MAX_SEG], seg_cpbegin[MG_MAX_SEG];
  int kv_per_tap, nkv, n_stages, n_tile, n_tiles;
  int n_rows_valid;  // forward: Cout; transposed: CcatP (rows that may be non-zero)
  int halo;          // stage order of the halo kernels: per chunk ceil(9 / tps) stages of tps taps each
  int stem;          // stage order of umma_stem_kernel: stage = kernel row ky, k-vector = (column pair q, parity): tap kx = 2q + parity
  int n_chunks;
  HChunk chunk[MAX_CHUNKS];
};

// one thread per (n row, k-vector): writes 16 bytes of the swizzled stage image
__device__ __forceinline__ void pack_one(const PackParams& p, int64_t i) {
  const int kv_total = p.n_stages * KV_PER_STAGE;
  const int64_t total = (int64_t)p.n_tiles * p.n_tile * kv_total;
  if (i >= total) return;
  const int j = (int)(i % kv_total);
  const int nrow = (int)(i / kv_total);          // global row = tile * n_tile + local
  const int tile = nrow / p.n_tile, nl = nrow % p.n_tile;
  const int stage = j / KV_PER_STAGE, v = j % KV_PER_STAGE;
  __nv_bfloat16 vals[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) vals[e] = __float2bfloat16_rn(0.f);
  const int KK = p.k * p.k;
  int tap, r, sg = 0, c0 = 0;   // tap, k-vector within the tap (generic order), K segment and first channel within it
  bool kv_ok;
  if (p.stem) {
    tap = stage * p.k + v;          // v = 2q + parity = kx (kx = 7 does not exist: zero column)
    kv_ok = v < p.k;
    sg = 0; c0 = 0; r = 0;
  } else if (p.halo) {
    int c = 0;
    while (c + 1 < p.n_chunks && stage >= p.chunk[c + 1].stage0) ++c;
    const HChunk ch = p.chunk[c];
    const int per = KV_PER_STAGE / ch.tps;        // k-vectors per tap within a stage
    tap = (stage - ch.stage0) * ch.tps + v / per;
    const int cv = v % per;
    kv_ok = tap < KK && cv * 8 < ch.nch;
    sg = ch.seg; c0 = ch.c0 + cv * 8;
    r = 0;
  } else {
    tap = j / p.kv_per_tap; r = j % p.kv_per_tap; kv_ok = j < p.nkv;
    if (!p.transposed) { while (sg + 1 < p.n_seg && r >= p.seg_kvbegin[sg + 1]) ++sg; c0 = (r - p.seg_kvbegin[sg]) * 8; }
    else c0 = r * 8;
  }
  if (kv_ok && nrow < p.n_rows_valid) {
    if (!p.transposed) {
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (c0 + e < p.seg_C[sg]) vals[e] = __float2bfloat16_rn(p.w[((size_t)nrow * p.Ccat + p.seg_cbegin[sg] + c0 + e) * KK + tap]);
    } else {
      // row = padded concat channel, K = (mirrored tap, output channel co)
      int rs = 0;
      while (rs + 1 < p.n_seg && nrow >= p.seg_cpbegin[rs + 1]) ++rs;
      const int cl = nrow - p.seg_cpbegin[rs];
      if (cl < p.seg_C[rs]) {
        const int ci = p.seg_cbegin[rs] + cl;
        const int ky = p.k - 1 - tap / p.k, kx = p.k - 1 - tap % p.k;
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (c0 + e < p.Cout) vals[e] = __float2bfloat16_rn(p.w[((size_t)(c0 + e) * p.Ccat + ci) * KK + ky * p.k + kx]);
      }
    }
  }
  uint8_t* dst = p.out + ((size_t)(tile * p.n_stages + stage) * p.n_tile + nl) * 128 + ((v ^ (nl & 7)) << 4);
  *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(vals);
}

__global__ void pack_weights_kernel(PackParams p) {
  pdl_launch();
  pdl_wait();
  pack_one(p, (int64_t)blockIdx.x * blockDim.x + threadIdx.x);
}

// every convolution of a plan in ONE launch: block b serves job j with blk_begin[j] <= b < blk_begin[j+1]
// (150 launches of ~4 us each, pure launch latency, become one HBM-bound pass)
__global__ void __launch_bounds__(256) pack_weights_batched_kernel(const PackParams* __restrict__ jobs, const int* __restrict__ blk_begin, int n_jobs) {
  pdl_launch();
  pdl_wait();
  int lo = 0, hi = n_jobs - 1;
  const int b = (int)blockIdx.x;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (blk_begin[mid] <= b) lo = mid; else hi = mid - 1;
  }
  __shared__ PackParams sp;
  const int* src = reinterpret_cast<const int*>(jobs + lo);
  for (int t = threadIdx.x; t < (int)(sizeof(PackParams) / sizeof(int)); t += blockDim.x) reinterpret_cast<int*>(&sp)[t] = src[t];
  __syncthreads();
  pack_one(sp, (int64_t)(b - blk_begin[lo]) * blockDim.x + threadIdx.x);
}

// ---------------------------------------------------------------- host side -----------------
struct Geometry {
  int kv_per_tap, nkv, n_stages, n_tile, n_tiles, n_rows;
  int halo, n_chunks, stem;
  HChunk chunk[MAX_CHUNKS];
};

// K of a halo convolution as chunks of <= 64 channels of ONE source grid (a TMA box never spans two grids); a chunk of
// <= 32 (<= 16) channels packs 2 (4) taps per 128-byte-row weight stage.  Returns the chunk count (> MAX_CHUNKS: no halo path)
static int build_chunks(const int* kcp, int nk, HChunk* out, int* n_stages) {
  int n = 0, st = 0;
  for (int s = 0; s < nk; ++s)
    for (int c0 = 0; c0 < kcp[s]; c0 += 64) {
      if (n == MAX_CHUNKS) return MAX_CHUNKS + 1;
      HChunk& ch = out[n++];
      ch.seg = s; ch.c0 = c0; ch.nch = std::min(64, kcp[s] - c0);
      ch.tps = ch.nch > 32 ? 1 : (ch.nch > 16 ? 2 : 4);
      ch.ksteps = (ch.nch + 15) / 16;
      ch.stage0 = st;
      st += (9 + ch.tps - 1) / ch.tps;
    }
  *n_stages = st;
  return n;
}

// the dedicated stem kernel: 7x7 / stride 2 / pad 3 on one image grid of <= 8 channels (Cp = 8), up to 256 output channels
static bool stem_shape_ok(const mg_conv_desc* d) {
  static int on = -1;
  if (on < 0) { const char* e = getenv("MGCONV_STEM_KERNEL"); on = e ? atoi(e) : 1; }
  if (!on || d->ksize != 7 || d->stride != 2 || d->pad != 3 || d->n_seg != 1 || d->seg_mode[0] != MG_SEG_SAME) return false;
  const mg_grid& g = d->seg[0];
  if (g.Cp != 8 || g.H != d->H || g.W != d->W || d->Cout > 256) return false;
  const int n_tile = mg_round_up(d->Cout, 16);
  return 7 * n_tile * 128 + 2 * (ST_SLOT + ST_RAW) + n_tile * 260 + 2048 <= 232448 - 4096;
}

static void n_tiling(int n_rows_pad16, int* n_tile, int* n_tiles) {
  *n_tiles = (n_rows_pad16 + 255) / 256;
  *n_tile = mg_round_up((n_rows_pad16 + *n_tiles - 1) / *n_tiles, 16);
}

// the halo kernels serve 3x3 / stride 1 / pad 1 convolutions on grids of at least `MGCONV_HALO_MIN_W`
// (default 7) and at most 64 columns whose UP segments are exactly half size
static bool halo_shape_ok(const mg_conv_desc* d) {
  static int min_w = -1;
  if (min_w < 0) { const char* e = getenv("MGCONV_HALO_MIN_W"); min_w = e ? atoi(e) : 7; }
  if (d->ksize != 3 || d->stride != 1 || d->pad != 1) return false;
  if (d->W < min_w || d->W > 64 || d->H > 1023) return false;
  for (int s = 0; s < d->n_seg; ++s) {
    const mg_grid& g = d->seg[s];
    if (d->seg_mode[s] == MG_SEG_UP) { if (g.H * 2 != d->H || g.W * 2 != d->W) return false; }
    else if (g.H != d->H || g.W != d->W) return false;
  }
  return (int64_t)d->seg[0].N * (d->H + 1) * (d->W + 1) < ((int64_t)1 << 31);
}

// geometry of the forward (transposed = 0) or dgrad (transposed = 1) GEMM of a conv descriptor
static Geometry geometry(const mg_conv_desc* d, int transposed) {
  Geometry g;
  memset(&g, 0, sizeof(g));
  int CcatP = 0;
  for (int s = 0; s < d->n_seg; ++s) CcatP += d->seg[s].Cp;
  const int CoutP = mg_round_up(d->Cout, 8);
  const int taps = d->ksize * d->ksize;
  if (!transposed) { g.kv_per_tap = CcatP / 8; g.n_rows = d->Cout; n_tiling(mg_round_up(d->Cout, 16), &g.n_tile, &g.n_tiles); }
  else { g.kv_per_tap = CoutP / 8; g.n_rows = CcatP; n_tiling(mg_round_up(CcatP, 16), &g.n_tile, &g.n_tiles); }
  g.nkv = taps * g.kv_per_tap;
  g.n_stages = (g.nkv + KV_PER_STAGE - 1) / KV_PER_STAGE;
  g.halo = 0;
  g.stem = 0;
  if (!transposed && stem_shape_ok(d)) { g.stem = 1; g.n_stages = 7; return g; }
  if (halo_shape_ok(d)) {
    int kcp[MG_MAX_SEG], nk, n_st = 0;
    if (!transposed) { nk = d->n_seg; for (int s = 0; s < nk; ++s) kcp[s] = d->seg[s].Cp; }
    else { nk = 1; kcp[0] = CoutP; }
    const int nc = build_chunks(kcp, nk, g.chunk, &n_st);
    if (nc <= MAX_CHUNKS) { g.halo = 1; g.n_chunks = nc; g.n_stages = n_st; }
  }
  return g;
}

static int pick_stages(int n_tile, int* smem_bytes) {
  const int stage = A_STAGE_BYTES + n_tile * 128;
  static int forced = -1;
  if (forced < 0) { const char* e = getenv("MGCONV_STAGES"); forced = e ? atoi(e) : 0; }
  static int budget_kb = -1;   // per-CTA shared memory target: ~54 KB keeps four CTAs resident per SM (measured best on R-MG-34)
  if (budget_kb < 0) { const char* e = getenv("MGCONV_SMEM_KB"); budget_kb = e ? atoi(e) : 54; }
  int S = forced > 0 ? forced : std::min(MAX_STAGES, (budget_kb * 1024) / stage);
  S = std::max(2, std::min(S, MAX_STAGES));
  *smem_bytes = S * stage + 1024;  // + alignment slack
  return S;
}

static int launch(mg_ctx* ctx, UParams& p, int n_tiles) {
  int smem = 0;
  p.stages = pick_stages(p.n_tile, &smem);
  p.stages = std::min(p.stages, std::max(2, p.n_stages));
  p.lag = std::max(0, std::min(p.stages - 2, 3));   // lag <= S-2: loaders issue ahead while the MMAs of the current stage run
  int cols = 32;
  while (cols < p.n_tile) cols <<= 1;
  p.tmem_cols = cols;
  static bool attr_set = false;
  if (!attr_set) {
    MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8 * 1024));
    MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8 * 1024));
    attr_set = true;
  }
  dim3 grid((unsigned)mg_cdiv(p.M, BM), (unsigned)n_tiles);
  // fast gather: stride 1, "same" padding (output size = input size), 1x1 or 3x3, every UP segment at exactly half size
  bool fast = p.stride == 1 && (p.k == 1 || p.k == 3) && p.pad == p.k / 2 && p.Ho == p.H && p.Wo == p.W && p.M < (int64_t)1 << 31;
  for (int s = 0; s < p.n_seg; ++s) {
    if (p.seg[s].shift) fast = fast && p.seg[s].Hs == p.H / 2 && p.seg[s].Ws == p.W / 2 && p.H % 2 == 0 && p.W % 2 == 0;
    else fast = fast && p.seg[s].Hs == p.H && p.seg[s].Ws == p.W;
  }
  if (fast) umma_conv_kernel<true><<<grid, N_THREADS, smem, ctx->stream>>>(p);
  else umma_conv_kernel<false><<<grid, N_THREADS, smem, ctx->stream>>>(p);
  MG_CHECK_LAUNCH(ctx);
  ctx->tc_launches++;
  return MG_OK;
}

constexpr int SMEM_MAX = 232448 - 4096;   // 227 KB per CTA minus the halo kernels' static shared memory (barriers, bias tile)

// halo geometry of a tile of `slots` GEMM rows on a grid of width W
static void halo_geometry(HParams& p, int slots) {
  p.HL = slots + 2 * p.Wp + 2;
  p.nr_max = (p.HL - 1 + p.Wp - 1) / p.Wp + 1;
  p.halo_bytes = mg_round_up((p.img_box ? p.HL : p.nr_max * p.Wp) * 128, 1024);
}

// whole-image TMA boxes: images of (H+1)*(W+1) slots that divide the tile (7 x 7 grids), no up-sampled segment
static bool img_box_ok(const HParams& p, int slots) {
  static int on = -1;
  if (on < 0) { const char* e = getenv("MGCONV_IMG_BOX"); on = e ? atoi(e) : 1; }
  const int spi = p.Hp * p.Wp;
  return on && !p.any_up && slots % spi == 0 && slots / spi <= 256;
}

// (re)build the tensor maps of the K segments for the tile size at hand
static int halo_tensor_maps(mg_ctx* ctx, HParams& p, const mg_grid* segs, int slots) {
  p.img_box = img_box_ok(p, slots) ? 1 : 0;
  for (int s = 0; s < p.n_seg; ++s) {
    const mg_grid& g = segs[s];
    int rc = p.img_box ? mg_tensor_map(ctx, g.data, p.Nimg, g.H, g.W, g.Cp, 4, slots / (p.Hp * p.Wp), &p.tmap[s])
                       : mg_tensor_map(ctx, g.data, p.Nimg, g.H, g.W, g.Cp, p.seg_up[s] ? 1 : 0, p.seg_up[s] ? 2 * g.W : p.Wp, &p.tmap[s]);
    if (rc) return rc;
  }
  return MG_OK;
}

// staging area of the bulk-store epilogue: behind the statistics scratch, if the CTA's shared memory (free once the MMAs are done)
// holds 128 * MT rows of n_tile * 2 + 16 bytes; returns byte offset + 1, or 0 for direct stores (MGCONV_EPI_STAGE=0)
static int epilogue_staging(const HParams& p, int MT, int smem_usable) {
  static int on = -1;
  if (on < 0) { const char* e = getenv("MGCONV_EPI_STAGE"); on = e ? atoi(e) : 1; }
  if (!on) return 0;
  const int off = p.stats ? MT * 4 * 2 * 256 * 4 : 0;
  const int need = off + MT * BM * (p.n_tile * 2 + 16);
  return need <= smem_usable ? off + 1 : 0;
}

static int launch_halo(mg_ctx* ctx, HParams& p, const Geometry& g, int algo, const mg_grid* segs) {
  const int b_stage = p.n_tile * 128;
  static int budget_env = -1, mt_env = -1;
  if (budget_env < 0) { const char* e = getenv("MGCONV_HALO_SMEM_KB"); budget_env = e ? atoi(e) : 0; }
  if (mt_env < 0) { const char* e = getenv("MGCONV_MT"); mt_env = e ? atoi(e) : 0; }
  // two sub-tiles per CTA (half the weight stream per row) whenever that still leaves about a CTA per SM
  int MT;
  {
    const int64_t ctas2 = mg_cdiv(p.T, 2 * BM) * g.n_tiles;
    const int want = (algo == MG_ALGO_TILE128 || algo == MG_ALGO_TILE128_DEEP || algo == MG_ALGO_TILE128_MID) ? 1
                     : ((algo == MG_ALGO_TILE256 || algo == MG_ALGO_TILE256_DEEP) ? 2 : (ctx->tune_mt ? ctx->tune_mt : mt_env));
    // heuristic: sharing the weight stages pays off once the K loop is long enough to amortise the bigger halo
    const bool heur2 = g.n_chunks >= 3 && ctas2 * 10 >= (int64_t)ctx->num_sms * 8;
    MT = (want == 1 || want == 2) ? want : (heur2 ? 2 : 1);
  }
  const bool pair = algo == MG_ALGO_PAIR128 || algo == MG_ALGO_PAIR256;
  if (pair) MT = algo == MG_ALGO_PAIR256 ? 2 : 1;
  { int rc = halo_tensor_maps(ctx, p, segs, BM * MT); if (rc) return rc; }
  halo_geometry(p, BM * MT);
  int cols = 32;
  while (cols < MT * p.n_tile) cols <<= 1;
  p.tmem_cols = cols;
  if (pair) {
    // CTA pairs (cta_group::2): half a weight stage per CTA; rows land up to Wp slots into the halo buffer (see the kernel)
    if (!p.img_box) p.halo_bytes = mg_round_up((p.nr_max * p.Wp + p.Wp) * 128, 1024);
    const int half = b_stage / 2;
    const int ctas = std::max(1, std::min(512 / cols, 2));
    int budget = (budget_env > 0 ? budget_env : (ctas == 1 ? 200 : 108)) * 1024;
    p.n_abuf = (g.n_chunks > 1 && 2 * p.halo_bytes + 2 * half <= budget) ? 2 : 1;
    int S = (budget - p.n_abuf * p.halo_bytes) / half;
    S = std::max(2, std::min(S, std::min(MAX_STAGES, p.n_stages)));
    p.stages = S;
    const int smem = p.n_abuf * p.halo_bytes + S * half + 1024;
    MG_REQUIRE(ctx, smem <= SMEM_MAX, MG_ERR_UNSUPPORTED, "pair halo conv: %d bytes of shared memory", smem);
    p.epi_stage = epilogue_staging(p, MT, smem - 1024);
    int rc = mg_tensor_map(ctx, p.wpack, g.n_tiles * p.n_stages * p.n_tile, 0, 0, 0, 5, p.n_tile / 2, &p.tmap_w);
    if (rc) return rc;
    static bool pair_attr_set = false;
    if (!pair_attr_set) {
      MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_halo_pair_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
      MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_halo_pair_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
      pair_attr_set = true;
    }
    dim3 grid((unsigned)mg_round_up((int)mg_cdiv(p.T, BM * MT), 2), (unsigned)g.n_tiles);   // an odd tile count gets an all-padding tile
    if (MT == 2) MG_CUDA(ctx, mg_launch_pdl(umma_conv_halo_pair_kernel<2>, grid, dim3(32 * 11), (size_t)smem, ctx->stream, p));
    else MG_CUDA(ctx, mg_launch_pdl(umma_conv_halo_pair_kernel<1>, grid, dim3(32 * 7), (size_t)smem, ctx->stream, p));
    MG_CHECK_LAUNCH(ctx);
    ctx->tc_launches++;
    return MG_OK;
  }
  int budget_kb;
  if (MT == 1) {
    // narrow tiles want several resident CTAs (prologue / epilogue of one overlap the main loop of the others);
    // N >= 192 tiles prefer two CTAs with a deeper weight ring
    budget_kb = p.n_tile >= 192 ? 108 : 56;
  } else {
    // TMEM allows 512 / cols CTAs per SM; at most two
    const int ctas = std::max(1, std::min(512 / cols, 2));
    budget_kb = ctas == 1 ? 200 : 108;
  }
  if (algo == MG_ALGO_TILE128_MID) budget_kb = 72;
  // grids with at most one CTA per SM (7 x 7 layers: 128 tiles) gain nothing from co-resident CTAs: every CTA streams the whole
  // weight image through its own ring, so give that ring all the shared memory there is (up to MAX_STAGES stages in flight)
  if ((algo == MG_ALGO_AUTO || algo == MG_ALGO_RESIDENT) && mg_cdiv(p.T, BM * MT) * g.n_tiles <= ctx->num_sms) budget_kb = 200;
  // "deep" variants trade resident CTAs for two halo buffers and a longer weight ring (more bytes in flight per CTA)
  if (algo == MG_ALGO_TILE128_DEEP) budget_kb = 108;
  if (algo == MG_ALGO_TILE256_DEEP) budget_kb = 200;
  if (budget_env > 0) budget_kb = budget_env;
  // two halo buffers when several chunks follow each other and the budget allows, else one
  const int min_ring = 2;
  p.n_abuf = (g.n_chunks > 1 && 2 * p.halo_bytes + min_ring * b_stage <= budget_kb * 1024) ? 2 : 1;
  int S = (budget_kb * 1024 - p.n_abuf * p.halo_bytes) / b_stage;
  S = std::max(2, std::min(S, std::min(MAX_STAGES, p.n_stages)));
  p.stages = S;
  static bool attr_set = false;
  if (!attr_set) {
    MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_halo_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
    MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_halo_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
    attr_set = true;
  }
  const int smem = p.n_abuf * p.halo_bytes + S * b_stage + 1024;
  MG_REQUIRE(ctx, smem <= SMEM_MAX, MG_ERR_UNSUPPORTED, "halo conv: %d bytes of shared memory", smem);
  p.epi_stage = epilogue_staging(p, MT, smem - 1024);
  dim3 grid((unsigned)mg_cdiv(p.T, BM * MT), (unsigned)g.n_tiles);
  if (MT == 2) MG_CUDA(ctx, mg_launch_pdl(umma_conv_halo_kernel<2>, grid, dim3(32 * 11), (size_t)smem, ctx->stream, p));
  else MG_CUDA(ctx, mg_launch_pdl(umma_conv_halo_kernel<1>, grid, dim3(32 * 7), (size_t)smem, ctx->stream, p));
  MG_CHECK_LAUNCH(ctx);
  ctx->tc_launches++;
  return MG_OK;
}

// shared-memory plan of the persistent kernel, or false when the weights do not fit / the launch is too small to pay off
struct PersistPlan { int n_abuf, smem, tmem_cols, grid, tile_rows, halo_bytes, pair; };
// row-aligned tiles of the persistent kernel: R whole slot rows per tile when they fill at least 85 % of the 128 MMA rows
static int persist_tile_rows(const mg_conv_desc* d, int Nimg, bool any_up) {
  const int Wp = d->W + 1, Hp = d->H + 1;
  if (Wp > BM) return 0;
  if (!any_up && BM % (Hp * Wp) == 0) return 0;          // whole-image boxes (7 x 7 grids) are better still
  const int R = BM / Wp;
  if (R < 1 || R * Wp * 100 < BM * 85) return 0;
  (void)Nimg;
  return R;
}
static bool persist_plan(const mg_ctx* ctx, const mg_conv_desc* d, const Geometry& g, int Nimg, int algo, bool stats, PersistPlan* pl) {
  static int on = -1, min_tiles_per_sm = -1;
  if (on < 0) { const char* e = getenv("MGCONV_PERSIST"); on = e ? atoi(e) : 1; }
  if (min_tiles_per_sm < 0) { const char* e = getenv("MGCONV_PERSIST_MIN_TILES"); min_tiles_per_sm = e ? atoi(e) : 4; }
  if (algo == MG_ALGO_TILE128 || algo == MG_ALGO_TILE256 || algo == MG_ALGO_TILE128_DEEP || algo == MG_ALGO_TILE256_DEEP ||
      algo == MG_ALGO_TILE128_MID || algo == MG_ALGO_PAIR128 || algo == MG_ALGO_PAIR256) return false;
  const bool pair = algo == MG_ALGO_RESIDENT_PAIR;
  const bool forced = algo == MG_ALGO_RESIDENT || pair || ctx->tune_persist == 1;
  if (!forced && (ctx->tune_persist == 2 || !on)) return false;
  if (!g.halo || g.n_tiles != 1) return false;
  HParams hp;
  hp.Wp = d->W + 1; hp.img_box = 0;     // sized for the row mode (the whole-image mode needs no more)
  halo_geometry(hp, BM);
  bool any_up = false;
  for (int s = 0; s < d->n_seg; ++s) any_up = any_up || d->seg_mode[s] == MG_SEG_UP;
  // row-aligned tiles: always for CTA pairs (same tile offset in both CTAs); for the single-CTA kernel only on request -- its
  // ring stays two tiles short either way and 12 % more tiles cost more than the smaller halo saves (measured: 125 -> 133 us).
  // Never when the epilogue reduces BatchNorm statistics: each warp sums its 32 slots in fp32 before the exact fixed-point total,
  // and only 128-slot tiles give every warp the same 32 slots in every variant; with R * Wp-slot tiles the statistics (and all
  // that follows them) would depend on which variant the autotuner timed fastest.
  static int aligned_single = -1;
  if (aligned_single < 0) { const char* e = getenv("MGCONV_PERSIST_ALIGNED"); aligned_single = e ? atoi(e) : 0; }
  const int R = ((pair || aligned_single) && !stats) ? persist_tile_rows(d, Nimg, any_up && g.n_chunks > 0) : 0;
  if (R) hp.halo_bytes = mg_round_up(((R + 2) * hp.Wp + 2) * 128, 1024);
  const int64_t m_tiles = R ? mg_cdiv((int64_t)Nimg * (d->H + 1), R) : mg_cdiv((int64_t)Nimg * (d->H + 1) * hp.Wp, BM);
  if (!forced && m_tiles < (int64_t)min_tiles_per_sm * ctx->num_sms) return false;
  if (pair && !R && !(!any_up && BM % ((d->H + 1) * hp.Wp) == 0)) return false;   // CTA pairs need the same tile offset in both CTAs
  const int b_bytes = g.n_stages * g.n_tile * (pair ? 64 : 128);                  // a pair keeps half of every stage per CTA
  const int tail = g.n_tile * (4 + 256);                   // bias tile + statistics accumulators (8 warps x 2 sums x 2 int64 limbs)
  const int room = SMEM_MAX - 1024 - b_bytes - tail;
  int n_abuf = room / hp.halo_bytes;
  if (n_abuf < 2) return false;
  n_abuf = std::min(n_abuf, std::min(P_MAX_ABUF, 2 * g.n_chunks + 1));
  int cols = 32;
  while (cols < 2 * g.n_tile) cols <<= 1;                  // two accumulators
  if (cols > 512) return false;
  pl->n_abuf = n_abuf; pl->smem = n_abuf * hp.halo_bytes + b_bytes + tail + 1024; pl->tmem_cols = cols;
  pl->grid = (int)std::min<int64_t>(m_tiles, ctx->num_sms);
  if (pair) pl->grid = 2 * (int)std::min<int64_t>((m_tiles + 1) / 2, ctx->num_sms / 2);
  pl->tile_rows = R; pl->halo_bytes = hp.halo_bytes; pl->pair = pair ? 1 : 0;
  return true;
}

static int launch_halo_persistent(mg_ctx* ctx, HParams& p, const PersistPlan& pl, const mg_grid* segs) {
  { int rc = halo_tensor_maps(ctx, p, segs, BM); if (rc) return rc; }
  halo_geometry(p, BM);
  p.m_tiles = (int)mg_cdiv(p.T, BM);
  p.tile_rows = p.img_box ? 0 : pl.tile_rows;
  if (p.tile_rows) {
    p.halo_bytes = pl.halo_bytes;
    p.nr_max = p.tile_rows + 2;
    p.m_tiles = (int)mg_cdiv((int64_t)p.Nimg * p.Hp, p.tile_rows);
  }
  p.tmem_cols = pl.tmem_cols;
  p.n_abuf = pl.n_abuf;
  p.stages = 0;
  static bool attr_set = false;
  if (!attr_set) {
    MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_halo_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
    attr_set = true;
  }
  if (pl.pair) {
    int rc = mg_tensor_map(ctx, p.wpack, p.n_stages * p.n_tile, 0, 0, 0, 5, p.n_tile / 2, &p.tmap_w);
    if (rc) return rc;
    static bool pair_attr = false;
    if (!pair_attr) {
      MG_CUDA(ctx, cudaFuncSetAttribute(umma_conv_halo_persistent_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX));
      pair_attr = true;
    }
    MG_CUDA(ctx, mg_launch_pdl(umma_conv_halo_persistent_pair_kernel, dim3(pl.grid), dim3(P_THREADS), (size_t)pl.smem, ctx->stream, p));
    MG_CHECK_LAUNCH(ctx);
    ctx->tc_launches++;
    return MG_OK;
  }
  MG_CUDA(ctx, mg_launch_pdl(umma_conv_halo_persistent_kernel, dim3(pl.grid), dim3(P_THREADS), (size_t)pl.smem, ctx->stream, p));
  MG_CHECK_LAUNCH(ctx);
  ctx->tc_launches++;
  return MG_OK;
}

static bool fused_stats_on() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("MGCONV_FUSED_STATS"); on = e ? atoi(e) : 1; }
  return on != 0;
}

// common part of the halo launches: geometry, chunk table and the tensor maps of the K segments (forward: the conv's source
// grids; dgrad: the gradient grid)
static int fill_halo_params(mg_ctx* ctx, HParams& p, const Geometry& g, int n_seg, const mg_grid* segs, const int* up, int N, int H, int W) {
  memset(&p, 0, sizeof(p));
  p.n_seg = n_seg; p.n_chunks = g.n_chunks; p.n_stages = g.n_stages;
  for (int c = 0; c < g.n_chunks; ++c) p.chunk[c] = g.chunk[c];
  p.H = H; p.W = W; p.Wp = W + 1; p.Hp = H + 1; p.Nimg = N;
  p.T = (int64_t)N * p.Hp * p.Wp;
  p.n_tile = g.n_tile;
  for (int s = 0; s < n_seg; ++s) {
    p.seg_up[s] = up[s];
    if (up[s]) p.any_up = 1;
  }
  return MG_OK;
}

}  // namespace

bool umma_wgrad_supported(const mg_ctx* ctx, const mg_conv_desc* d);

bool umma_conv_supported(const mg_ctx* ctx, const mg_conv_desc* d, int kind) {
  if (ctx->dtype != MG_BF16) return false;
  if (kind == 2) return umma_wgrad_supported(ctx, d);
  if (kind == 1 && d->stride != 1) return false;     // dgrad of the strided stem is never needed
  if (d->n_seg < 1 || d->n_seg > MG_MAX_SEG) return false;
  for (int s = 0; s < d->n_seg; ++s) {
    const mg_grid& g = d->seg[s];
    if (d->seg_mode[s] == MG_SEG_POOL) return false;  // gathers are pure copies: POOL operands come as pooled companions
    if (g.scale || g.shift) return false;             // pending affines are materialised by the apply pass
    if (g.Cp % 8) return false;
    if (g.H > 1023 || g.W > 1023 || g.N > 4095) return false;
  }
  return d->H <= 1023 && d->W <= 1023;
}

size_t umma_packed_bytes(const mg_conv_desc* d, int transposed) {
  if (!d || d->n_seg < 1 || d->n_seg > MG_MAX_SEG) return 0;
  if (transposed && d->stride != 1) return 0;
  for (int s = 0; s < d->n_seg; ++s)
    if (d->seg_mode[s] == MG_SEG_POOL || d->seg[s].scale || d->seg[s].Cp % 8) return 0;
  Geometry g = geometry(d, transposed);
  return (size_t)g.n_tiles * g.n_stages * g.n_tile * 128;
}

static PackParams make_pack_params(const mg_conv_desc* d, const float* w, void* wpack, int transposed, int64_t* total) {
  Geometry g = geometry(d, transposed);
  PackParams p;
  memset(&p, 0, sizeof(p));
  p.w = w; p.out = (uint8_t*)wpack; p.transposed = transposed;
  p.k = d->ksize; p.Cout = d->Cout; p.n_seg = d->n_seg;
  int c = 0, cp = 0;
  for (int s = 0; s < d->n_seg; ++s) {
    p.seg_C[s] = d->seg[s].C; p.seg_cbegin[s] = c; p.seg_cpbegin[s] = cp; p.seg_kvbegin[s] = cp / 8;
    c += d->seg[s].C; cp += d->seg[s].Cp;
  }
  p.Ccat = c;
  p.kv_per_tap = g.kv_per_tap; p.nkv = g.nkv; p.n_stages = g.n_stages; p.n_tile = g.n_tile; p.n_tiles = g.n_tiles;
  p.n_rows_valid = g.n_rows; p.halo = g.halo; p.stem = g.stem;
  p.n_chunks = g.n_chunks;
  for (int i = 0; i < g.n_chunks; ++i) p.chunk[i] = g.chunk[i];
  *total = (int64_t)g.n_tiles * g.n_tile * g.n_stages * KV_PER_STAGE;
  return p;
}

int umma_pack_weights(mg_ctx* ctx, const mg_conv_desc* d, const float* w, void* wpack, int transposed) {
  int64_t total = 0;
  PackParams p = make_pack_params(d, w, wpack, transposed, &total);
  mg_launch_pdl(pack_weights_kernel, dim3((unsigned)mg_cdiv(total, 256)), dim3(256), 0, ctx->stream, p);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// The job table lives in device memory owned by the context and is re-uploaded only when its contents change
// (plans are static: one upload, then every step is a single launch -- and nothing but that launch is seen by a
// CUDA-graph capture of the step).
int umma_pack_weights_batched(mg_ctx* ctx, int n, const mg_conv_desc* const* descs, const float* const* w, void* const* wpack,
                              const int32_t* transposed) {
  static_assert(sizeof(PackParams) % sizeof(int) == 0, "PackParams is copied as ints");
  std::vector<PackParams> jobs((size_t)n);
  std::vector<int> blk((size_t)n + 1);
  int64_t nb = 0;
  for (int j = 0; j < n; ++j) {
    MG_REQUIRE(ctx, descs[j] && w[j] && wpack[j], MG_ERR_INVALID_ARG, "pack_weights_batched: job %d has a null pointer", j);
    int64_t total = 0;
    jobs[j] = make_pack_params(descs[j], w[j], wpack[j], transposed[j], &total);
    blk[j] = (int)nb;
    nb += mg_cdiv(total, 256);
    MG_REQUIRE(ctx, nb < ((int64_t)1 << 31), MG_ERR_UNSUPPORTED, "pack_weights_batched: too many blocks");
  }
  blk[n] = (int)nb;
  const size_t jb = (size_t)n * sizeof(PackParams), bb = ((size_t)n + 1) * sizeof(int), bytes = jb + bb;
  std::vector<uint8_t> image(bytes);
  memcpy(image.data(), jobs.data(), jb);
  memcpy(image.data() + jb, blk.data(), bb);
  if (ctx->pack_bytes != bytes || !ctx->pack_host || memcmp(ctx->pack_host, image.data(), bytes) != 0) {
    if (ctx->pack_cap < bytes) {
      MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      if (ctx->pack_dev) cudaFree(ctx->pack_dev);
      free(ctx->pack_host);
      ctx->pack_dev = nullptr; ctx->pack_host = nullptr; ctx->pack_cap = 0; ctx->pack_bytes = 0;
      MG_CUDA(ctx, cudaMalloc(&ctx->pack_dev, bytes));
      ctx->pack_host = malloc(bytes);
      MG_REQUIRE(ctx, ctx->pack_host != nullptr, MG_ERR_INVALID_ARG, "pack_weights_batched: out of host memory");
      ctx->pack_cap = bytes;
    }
    memcpy(ctx->pack_host, image.data(), bytes);
    ctx->pack_bytes = bytes;
    // pageable source: staged by the driver before the call returns, ordered on the stream after earlier readers
    MG_CUDA(ctx, cudaMemcpyAsync(ctx->pack_dev, ctx->pack_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  const PackParams* djobs = (const PackParams*)ctx->pack_dev;
  const int* dblk = (const int*)((const uint8_t*)ctx->pack_dev + jb);
  if (nb > 0) {
    MG_CUDA(ctx, mg_launch_pdl(pack_weights_batched_kernel, dim3((unsigned)nb), dim3(256), 0, ctx->stream, djobs, dblk, n));
    MG_CHECK_LAUNCH(ctx);
  }
  return MG_OK;
}

int umma_conv_forward(mg_ctx* ctx, const mg_conv_desc* d, const void* wpack, const float* bias, mg_grid* y, mg_sum* bn_sums) {
  Geometry g = geometry(d, 0);
  int up[MG_MAX_SEG];
  for (int s = 0; s < d->n_seg; ++s) {
    const mg_grid& sg = d->seg[s];
    const int m = d->seg_mode[s];
    if (m == MG_SEG_SAME) MG_REQUIRE(ctx, sg.H == d->H && sg.W == d->W, MG_ERR_SHAPE, "conv: SAME seg %d is %dx%d, expected %dx%d", s, sg.H, sg.W, d->H, d->W);
    else MG_REQUIRE(ctx, sg.H * 2 == d->H && sg.W * 2 == d->W, MG_ERR_SHAPE, "conv: UP seg %d is %dx%d, x2 != %dx%d", s, sg.H, sg.W, d->H, d->W);
    MG_REQUIRE(ctx, sg.N == d->seg[0].N, MG_ERR_SHAPE, "conv: seg %d batch", s);
    up[s] = m == MG_SEG_UP ? 1 : 0;
  }
  if (g.stem) {
    StemParams sp;
    memset(&sp, 0, sizeof(sp));
    int rc = mg_tensor_map(ctx, d->seg[0].data, y->N, d->H, d->W, 8, 2, ST_RAW_COLS, &sp.tmap);
    if (rc) return rc;
    sp.H = d->H; sp.W = d->W; sp.Ho = y->H; sp.Wo = y->W; sp.Nimg = y->N;
    sp.tiles_x = (y->W + 7) / 8; sp.tiles_y = (y->H + 15) / 16;
    sp.n_tiles_total = y->N * sp.tiles_x * sp.tiles_y;
    sp.n_tile = g.n_tile;
    sp.wpack = (const uint8_t*)wpack; sp.bias = bias; sp.c_bias = d->Cout;
    sp.y = (__nv_bfloat16*)y->data; sp.y_pitch = y->Cp; sp.c_valid = y->Cp;
    // measured (B = 256, 224 x 224 -> 112 x 112 x 64): 210 us without the sums, 435 us with them fused in the epilogue (the four
    // warps per accumulator cannot keep up with a tile every ~1 200 cycles), 210 + 110 us with the separate statistics pass
    const bool fused = bn_sums && fused_stats_on() && ctx->tune_stem_fused;
    if (fused) { sp.stats = bn_sums; sp.c_stats = d->Cout; }
    int cols = 32;
    while (cols < 2 * g.n_tile) cols <<= 1;
    sp.tmem_cols = cols;
    sp.tma_out = (g.n_tile == 64 && y->Cp == 64) ? 1 : 0;
    if (sp.tma_out) { rc = mg_tensor_map(ctx, y->data, y->N, y->H, y->W, y->Cp, 3, 8, &sp.tmap_y); if (rc) return rc; }
    const int fixed = 7 * g.n_tile * 128 + g.n_tile * 260 + 1024 + (sp.tma_out ? 32768 : 0);
    sp.ring = std::max(2, std::min(ST_MAX_RING, (SMEM_MAX - fixed) / (ST_SLOT + ST_RAW)));
    static bool attr_set = false;
    if (!attr_set) { MG_CUDA(ctx, cudaFuncSetAttribute(umma_stem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_MAX)); attr_set = true; }
    const int grid = std::min(sp.n_tiles_total, ctx->num_sms);
    MG_CUDA(ctx, mg_launch_pdl(umma_stem_kernel, dim3(grid), dim3(ST_THREADS), (size_t)(fixed + sp.ring * (ST_SLOT + ST_RAW)), ctx->stream, sp));
    MG_CHECK_LAUNCH(ctx);
    ctx->tc_launches++;
    if (bn_sums && !fused) return mg_bn_stats(ctx, y, bn_sums);
    return MG_OK;
  }
  if (g.halo) {
    HParams hp;
    int rc = fill_halo_params(ctx, hp, g, d->n_seg, d->seg, up, y->N, d->H, d->W);
    if (rc) return rc;
    hp.wpack = (const uint8_t*)wpack; hp.bias = bias; hp.c_bias = d->Cout;
    hp.y = (__nv_bfloat16*)y->data; hp.y_pitch = y->Cp; hp.c_valid = y->Cp;
    // the halo kernels reduce the BatchNorm statistics in their epilogue; the other kernels are followed by the statistics pass
    const bool fused_stats = bn_sums && fused_stats_on();
    if (fused_stats) { hp.stats = bn_sums; hp.c_stats = d->Cout; }
    PersistPlan pl;
    rc = persist_plan(ctx, d, g, hp.Nimg, d->algo_fwd, hp.stats != nullptr, &pl) ? launch_halo_persistent(ctx, hp, pl, d->seg) : launch_halo(ctx, hp, g, d->algo_fwd, d->seg);
    if (rc) return rc;
    if (bn_sums && !fused_stats) return mg_bn_stats(ctx, y, bn_sums);
    return MG_OK;
  }
  UParams p;
  memset(&p, 0, sizeof(p));
  p.n_seg = d->n_seg;
  int cp = 0;
  for (int s = 0; s < d->n_seg; ++s) {
    const mg_grid& sg = d->seg[s];
    p.seg[s].ptr = (const __nv_bfloat16*)sg.data; p.seg[s].Hs = sg.H; p.seg[s].Ws = sg.W; p.seg[s].Cp = sg.Cp;
    p.seg[s].shift = up[s]; p.seg[s].kv_begin = cp / 8;
    cp += sg.Cp;
  }
  p.k = d->ksize; p.stride = d->stride; p.pad = d->pad; p.H = d->H; p.W = d->W;
  p.Ho = y->H; p.Wo = y->W; p.Nimg = y->N;
  p.M = (int64_t)y->N * y->H * y->W;
  p.kv_per_tap = g.kv_per_tap; p.nkv = g.nkv; p.n_stages = g.n_stages; p.n_tile = g.n_tile;
  p.wpack = (const uint8_t*)wpack; p.bias = bias; p.c_bias = d->Cout;
  p.y = (__nv_bfloat16*)y->data; p.y_pitch = y->Cp; p.c_valid = y->Cp;
  int rc = launch(ctx, p, g.n_tiles);
  if (rc) return rc;
  if (bn_sums) return mg_bn_stats(ctx, y, bn_sums);
  return MG_OK;
}

int umma_conv_backward_data(mg_ctx* ctx, const mg_conv_desc* d, const void* wpack_t, const mg_grid* gr, mg_grid* dcat) {
  Geometry g = geometry(d, 1);
  MG_REQUIRE(ctx, gr->Cp == mg_round_up(d->Cout, 8), MG_ERR_SHAPE, "dgrad: g.Cp %d", gr->Cp);
  MG_REQUIRE(ctx, dcat->Cp == g.n_rows, MG_ERR_SHAPE, "dgrad: dcat.Cp %d != %d", dcat->Cp, g.n_rows);
  if (g.halo) {
    HParams hp;
    const int up0 = 0;
    int rc = fill_halo_params(ctx, hp, g, 1, gr, &up0, dcat->N, gr->H, gr->W);
    if (rc) return rc;
    hp.wpack = (const uint8_t*)wpack_t; hp.bias = nullptr;
    hp.y = (__nv_bfloat16*)dcat->data; hp.y_pitch = dcat->Cp; hp.c_valid = dcat->Cp;
    PersistPlan pl;
    return persist_plan(ctx, d, g, hp.Nimg, d->algo_bwd_data, false, &pl) ? launch_halo_persistent(ctx, hp, pl, gr) : launch_halo(ctx, hp, g, d->algo_bwd_data, gr);
  }
  UParams p;
  memset(&p, 0, sizeof(p));
  p.n_seg = 1;
  p.seg[0].ptr = (const __nv_bfloat16*)gr->data; p.seg[0].Hs = gr->H; p.seg[0].Ws = gr->W; p.seg[0].Cp = gr->Cp;
  p.seg[0].shift = 0; p.seg[0].kv_begin = 0;
  p.k = d->ksize; p.stride = 1; p.pad = d->ksize - 1 - d->pad; p.H = gr->H; p.W = gr->W;
  p.Ho = dcat->H; p.Wo = dcat->W; p.Nimg = dcat->N;
  p.M = (int64_t)dcat->N * dcat->H * dcat->W;
  p.kv_per_tap = g.kv_per_tap; p.nkv = g.nkv; p.n_stages = g.n_stages; p.n_tile = g.n_tile;
  p.wpack = (const uint8_t*)wpack_t; p.bias = nullptr;
  p.y = (__nv_bfloat16*)dcat->data; p.y_pitch = dcat->Cp; p.c_valid = dcat->Cp;
  return launch(ctx, p, g.n_tiles);
}
