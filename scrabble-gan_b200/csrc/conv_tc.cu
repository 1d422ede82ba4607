// tcgen05 / TMEM / TMA implicit-GEMM convolution for sm_100a (K1-K7: the >=99% of step FLOPs).
//
// Reference ops replaced: Conv2D, Conv2DBackpropInput, Conv2DBackpropFilter, Conv2DTranspose as dispatched by
// resnet_ops.py:57,65,69,98,103,109 and net_architecture.py:28-49 (SURVEY.md section 2.2 K1-K7).
//
// Forward-type kernel (also serves dgrad and the transposed convs through the generic sg_conv_desc):
//   D[128 pixels, BN channels] = sum over (tap, 128-byte channel chunk) A_tap[128 pixels, KC] * W[BN, KC]^T
//   * A tile: ONE 4-D tiled TMA box (KC channels x TW x TH x TN pixels) per k-block, at the tap-shifted
//     coordinate; out-of-image pixels (SAME padding halo, ragged edges) are zero-filled by the TMA unit, so
//     there is no im2col buffer and no predication in the main loop.  Strided sampling (transposed-conv
//     dgrad) uses one tensor map per sampling phase.
//   * B tile: 2-D TMA box of the pre-packed K-major weight matrix [c_out][ntaps*c_in].
//   * both tiles land in 128B-swizzled shared memory and are consumed by tcgen05.mma (cta_group::1,
//     M=128, N=BN<=256, K=32 bytes) issued by one thread; fp32 accumulators live in TMEM, double-buffered so
//     the epilogue of tile i overlaps the main loop of tile i+1.
//   * warp roles: warp0 = TMA producer, warp1 = MMA issuer (+TMEM alloc), warps 2..5 = epilogue
//     (tcgen05.ld -> bias / ReLU / mask / accumulate -> vectorised global stores, NHWC, optional strided
//     placement for transposed-conv phases).
//   * persistent: grid = min(#tiles, #SMs), static round-robin tile schedule, N-tile fastest so that CTAs
//     running concurrently share the same activation tile through L2.
// Filter-gradient kernel: D[128 c_out, BN c_in] += dy_tile^T[128, P] * in_tile[P, BN] with BOTH operands
// MN-major (pixels are the reduction dim and the slow smem dim), split over pixel ranges with fp32 red.add.
#include "common.cuh"
#include <stdlib.h>

// ---------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spins = 0;; ++spins) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if (spins > (1u << 24)) __trap();     // a protocol bug must fault, never hang the GPU
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
template <bool kTf32>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kTf32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout SWIZZLE_128B=2 [61,64)
// layout 2 = SWIZZLE_128B (16-byte atoms), 1 = SWIZZLE_128B_BASE32B (32-byte atoms: the only layout for MN-major tf32)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = 2) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32=1 @4, a/b format @7/@10 (BF16=1, TF32=2),
// a_major @15, b_major @16 (0 = K-major, 1 = MN-major), N>>3 @17, M>>4 @24
__host__ __device__ inline uint32_t make_idesc(bool tf32, bool a_mn, bool b_mn, int m, int n) {
  uint32_t fmt = tf32 ? 2u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

#define TC_MAX_STAGES 8
#define TC_EPI_STAGING (4 * 32 * 33 * 4)      // per-warp 32 x 33 fp32 transpose buffers of the 4 epilogue warps
#define TC_THREADS 192
#define TC_TMEM_COLS 512

// ---------------------------------------------------------------------------------------------------
// forward-type kernel
// ---------------------------------------------------------------------------------------------------
struct alignas(64) TcFwdParams {
  CUtensorMap map_a[4];
  CUtensorMap map_b;
  CUtensorMap map_a2, map_b2;   // optional second (1x1) conv accumulated into the same tile: kc2 extra k-blocks (0 = none)
  int kc2;
  int tap_view[SG_MAX_TAPS], tap_oy[SG_MAX_TAPS], tap_ox[SG_MAX_TAPS];
  int tap_wt[SG_MAX_TAPS];      // direct-weight modes: index of tap t in the master filter (3rd TMA coordinate)
  int b_mode;                   // 0 = packed K-major matrix (2-D map); 1 = master read in place, K-major; 2 = in place, N-major
  int ntaps, c_in, c_out, n, grid_h, grid_w;
  int out_h, out_w, out_sy, out_sx, out_py, out_px;
  int TW, TH, TN, tiles_x, tiles_y, tiles_n, tiles_col, BN;
  int kc_per_tap, stages;
  uint32_t a_bytes, b_bytes, a_stage_stride, b_stage_stride;
  int relu, accumulate, out_dt, mask_dt;
  const float* bias;
  const void* mask;
  void* out;
  // optional rank-1 term of the epilogue: out[p, c] += r1_x[p] * r1_w[c] -- the 1x1 shortcut conv of a block whose input has ONE
  // channel (D.B1.short on the raw image, resnet_ops.py:107-110), which is an outer product, not a GEMM
  const float* r1_x;            // [n, out_h, out_w] fp32, indexed like the output pixels
  const float* r1_w;            // [c_out] fp32
  // split tail (wave quantisation): tiles [0, t_full) are whole units; each later tile is `split` units, one contiguous k-block
  // range each, on `split` consecutive CTAs.  Every unit parks the accumulator chunks it does not own in `part`, the units of a
  // tile meet at `cnt`, and each finishes its own share of the tile's 32-column chunks: own accumulators + the peers' partials
  // added in unit order (deterministic), then the usual epilogue.
  int t_full, split, total_units;
  // phases of a transposed conv in ONE launch (sg_conv_fwd_tc_phases): tile / tiles_per_phase selects the phase, which owns
  // taps [ph_tap0, ph_tap0 + ph_ntaps) of the tap tables and writes at output offset (ph_py, ph_px).  nphase == 1: plain conv.
  int nphase, tiles_per_phase;
  int ph_tap0[4], ph_ntaps[4], ph_py[4], ph_px[4];
  float* part;                  // [tail unit][BN/32 chunks][8][128 rows] float4
  unsigned int* cnt;            // [tail tile][2]: arrivals, departures; zero between launches
};

// unit v of the launch -> (tile inside its phase, phase, k-block range); si = index of the unit inside its tile (0 for whole tiles)
struct TcUnit { int tile, ph, kb0, kb1, si, tail_tile; };
__device__ __forceinline__ TcUnit tc_unit(const TcFwdParams& p, int v) {
  TcUnit u;
  int gt;                               // global tile index
  if (v < p.t_full) { gt = v; u.si = 0; u.tail_tile = -1; }
  else {
    const int w = v - p.t_full;
    gt = p.t_full + w / p.split;
    u.si = w % p.split;
    u.tail_tile = w / p.split;
  }
  u.ph = gt / p.tiles_per_phase;
  u.tile = gt - u.ph * p.tiles_per_phase;
  const int nkb = p.ph_ntaps[u.ph] * p.kc_per_tap + p.kc2;
  if (v < p.t_full) { u.kb0 = 0; u.kb1 = nkb; }
  else {
    u.kb0 = (int)((long long)nkb * u.si / p.split);
    u.kb1 = (int)((long long)nkb * (u.si + 1) / p.split);
  }
  return u;
}

template <typename TIn>
__global__ void __launch_bounds__(TC_THREADS, 1) k_conv_tc(const __grid_constant__ TcFwdParams p) {
  constexpr bool kTf32 = sizeof(TIn) == 4;
  constexpr int KC = 128 / sizeof(TIn);            // elements per 128-byte swizzle row
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * TC_MAX_STAGES + 4];
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + p.stages * p.a_stage_stride;
  const uint32_t bar_full = smem_u32(&bars[0]);
  const uint32_t bar_empty = smem_u32(&bars[TC_MAX_STAGES]);
  const uint32_t bar_tfull = smem_u32(&bars[2 * TC_MAX_STAGES]);
  const uint32_t bar_tempty = smem_u32(&bars[2 * TC_MAX_STAGES + 2]);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, 128);
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    for (int v = 0; v < 4; ++v) tma_prefetch_desc(&p.map_a[v]);
    tma_prefetch_desc(&p.map_b);
    if (p.kc2) { tma_prefetch_desc(&p.map_a2); tma_prefetch_desc(&p.map_b2); }
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_slot), TC_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int v = blockIdx.x; v < p.total_units; v += gridDim.x) {
        const TcUnit u = tc_unit(p, v);
        const int tile = u.tile;
        const int nkb1 = p.ph_ntaps[u.ph] * p.kc_per_tap;
        int col_t = tile % p.tiles_col, mt = tile / p.tiles_col;
        int tx = mt % p.tiles_x;
        int r = mt / p.tiles_x;
        int ty = r % p.tiles_y, tn = r / p.tiles_y;
        int x0 = tx * p.TW, y0 = ty * p.TH, n0 = tn * p.TN, col0 = col_t * p.BN;
        int t = p.ph_tap0[u.ph] + u.kb0 / p.kc_per_tap, c = u.kb0 % p.kc_per_tap;      // (tap, channel chunk) of k-block kb < nkb1
        for (int kb = u.kb0; kb < u.kb1; ++kb) {
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          mbar_expect_tx(bar_full + 8 * s, p.a_bytes + p.b_bytes);
          if (kb < nkb1) {
            const CUtensorMap* ma = &p.map_a[p.tap_view[t]];
            tma_load_4d(a_base + s * p.a_stage_stride, ma, bar_full + 8 * s, c * KC, x0 + p.tap_ox[t], y0 + p.tap_oy[t], n0);
            const uint32_t bdst = b_base + s * p.b_stage_stride;
            if (p.b_mode == 0) {
              tma_load_2d(bdst, &p.map_b, bar_full + 8 * s, t * p.c_in + c * KC, col0);
            } else if (p.b_mode == 1) {          // master [tap][c_out][c_in]: the same [BN rows][KC] K-major tile, read in place
              tma_load_3d(bdst, &p.map_b, bar_full + 8 * s, c * KC, col0, p.tap_wt[t]);
            } else {                             // master [tap][c_in][c_out]: N-major chunks of [KC rows][64 columns]
              for (int j = 0; j < p.BN / 64; ++j)
                tma_load_3d(bdst + j * (KC * 128), &p.map_b, bar_full + 8 * s, col0 + 64 * j, c * KC, p.tap_wt[t]);
            }
            if (++c == p.kc_per_tap) { c = 0; ++t; }
          } else {                               // second operand: the block's 1x1 shortcut on its own input tensor
            const int c2 = kb - nkb1;
            tma_load_4d(a_base + s * p.a_stage_stride, &p.map_a2, bar_full + 8 * s, c2 * KC, x0, y0, n0);
            tma_load_2d(b_base + s * p.b_stage_stride, &p.map_b2, bar_full + 8 * s, c2 * KC, col0);
          }
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const bool b_mn = p.b_mode == 2;
    const uint32_t idesc = make_idesc(kTf32, false, b_mn, 128, p.BN);
    int s = 0, as = 0;
    uint32_t ph = 0, aph = 0;
    for (int v = blockIdx.x; v < p.total_units; v += gridDim.x) {
      const TcUnit u = tc_unit(p, v);
      mbar_wait(bar_tempty + 8 * as, aph ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)as * 256u;
      for (int kb = u.kb0; kb < u.kb1; ++kb) {
        mbar_wait(bar_full + 8 * s, ph);
        tc_fence_after();
        if (lane == 0) {
          uint64_t da = make_smem_desc(a_base + s * p.a_stage_stride, 16, 1024);
          // K-major B: 32 bytes of K per step inside the 128-byte swizzle row.  N-major B (weights read in place):
          // LBO = distance between the 64-column chunks, a K step of 16 rows = 16 x 128 bytes.
          uint64_t db = b_mn ? make_smem_desc(b_base + s * p.b_stage_stride, KC * 128, 1024)
                             : make_smem_desc(b_base + s * p.b_stage_stride, 16, 1024);
          const uint64_t bstep = b_mn ? (uint64_t)((16 * 128) >> 4) : 2ull;
#pragma unroll
          for (int k = 0; k < 4; ++k)      // 4 x 32 bytes of K per 128-byte swizzle row of A
            umma<kTf32>(d_tmem, da + (uint64_t)(2 * k), db + bstep * k, idesc, (kb != u.kb0 || k != 0) ? 1u : 0u);
          umma_commit(bar_empty + 8 * s);
          if (kb == u.kb1 - 1) umma_commit(bar_tfull + 8 * as);
        }
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1; }
      }
      as ^= 1;
      if (as == 0) aph ^= 1;
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    // tcgen05.ld hands every lane ONE accumulator row (pixel) x 32 consecutive channels.  Storing that directly would
    // make each warp store touch 32 different pixels (32 sectors, 8..16 useful bytes each), so the 32 x 32 chunk goes
    // through a per-warp shared-memory transpose: afterwards 4 adjacent lanes own 32 consecutive channels of one pixel
    // (64 B of bf16 / 128 B of fp32 contiguous) and every store / mask load / accumulate load is sector-exact.
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may access
    const int row = quarter * 32 + lane;           // accumulator row = pixel index inside the tile
    const int rows_in_tile = p.TW * p.TH * p.TN;
    float* stg = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw)) + p.stages * (p.a_stage_stride + p.b_stage_stride)) +
                 (warp - 2) * (32 * 33);
    const int tr0 = lane >> 2, c0 = (lane & 3) * 8;      // transposed ownership: rows tr0 + 8 i, channels c0 .. c0 + 7
    int as = 0;
    uint32_t aph = 0;
    const int nchunks = p.BN / 32;
    for (int v = blockIdx.x; v < p.total_units; v += gridDim.x) {
      const TcUnit u = tc_unit(p, v);
      const int tile = u.tile;
      const int out_py = p.ph_py[u.ph], out_px = p.ph_px[u.ph];
      int col_t = tile % p.tiles_col, mt = tile / p.tiles_col;
      int tx = mt % p.tiles_x;
      int r = mt / p.tiles_x;
      int ty = r % p.tiles_y, tn = r / p.tiles_y;
      int ln = row / (p.TH * p.TW), rem = row % (p.TH * p.TW);
      int ly = rem / p.TW, lx = rem % p.TW;
      int ni = tn * p.TN + ln, oy = ty * p.TH + ly, ox = tx * p.TW + lx;
      bool valid = row < rows_in_tile && ni < p.n && oy < p.grid_h && ox < p.grid_w;
      long long base = -1;                                  // < 0 = no such output pixel
      if (valid)
        base = (((long long)ni * p.out_h + oy * p.out_sy + out_py) * p.out_w + ox * p.out_sx + out_px) * p.c_out +
               col_t * p.BN;
      long long rbase[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) rbase[i] = __shfl_sync(0xffffffffu, base, tr0 + 8 * i);
      const float r1 = (p.r1_x && valid) ? __ldg(p.r1_x + (base - col_t * p.BN) / p.c_out) : 0.f;
      mbar_wait(bar_tfull + 8 * as, aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)as * 256u;
      int ch_lo = 0, ch_hi = nchunks;
      const float4* peers = nullptr;                        // partials of the tile's units, unit 0 first
      if (v >= p.t_full) {
        // a split tile: park the chunks the peers will finish, meet them, then finish chunks [ch_lo, ch_hi) of the tile
        ch_lo = nchunks * u.si / p.split;
        ch_hi = nchunks * (u.si + 1) / p.split;
        const int tail_tile = u.tail_tile;
        const long long unit_f4 = (long long)nchunks * 8 * 128;
        peers = reinterpret_cast<const float4*>(p.part) + (long long)tail_tile * p.split * unit_f4;
        float4* mine = reinterpret_cast<float4*>(p.part) + ((long long)tail_tile * p.split + u.si) * unit_f4;
        for (int ch = 0; ch < nchunks; ++ch) {
          if (ch >= ch_lo && ch < ch_hi) continue;
          uint32_t pv[32];
          tmem_ld32(taddr + ch * 32, pv);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            __stcg(mine + ((long long)ch * 8 + j) * 128 + row,
                   make_float4(__uint_as_float(pv[4 * j]), __uint_as_float(pv[4 * j + 1]), __uint_as_float(pv[4 * j + 2]), __uint_as_float(pv[4 * j + 3])));
        }
        __threadfence();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        unsigned int* cn = p.cnt + 2 * tail_tile;
        if (threadIdx.x == 64) {
          atomicAdd(cn, 1u);
          unsigned int spins = 0;
          while (*reinterpret_cast<volatile unsigned int*>(cn) < (unsigned int)p.split) {
            if (++spins > (1u << 26)) __trap();          // a protocol bug must fault, never hang the GPU
            __nanosleep(64);
          }
          __threadfence();
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      for (int ch = ch_lo; ch < ch_hi; ++ch) {
        // issue every global read of this chunk (ReLU mask, accumulate operand) up front: all of them are in flight while
        // the accumulators come out of TMEM and go through the transpose
        float mk[4][8], prev[4][8];
        const bool want_prev = p.accumulate && p.out_dt == SG_F32;
        if (p.mask) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (rbase[i] < 0) continue;
            const long long off = rbase[i] + ch * 32 + c0;
            float4 a, b;
            if (p.mask_dt == SG_F32) {
              const float* mp = reinterpret_cast<const float*>(p.mask) + off;
              a = sg_ld4(mp); b = sg_ld4(mp + 4);
            } else {
              const __nv_bfloat16* mp = reinterpret_cast<const __nv_bfloat16*>(p.mask) + off;
              a = sg_ld4(mp); b = sg_ld4(mp + 4);
            }
            mk[i][0] = a.x; mk[i][1] = a.y; mk[i][2] = a.z; mk[i][3] = a.w; mk[i][4] = b.x; mk[i][5] = b.y; mk[i][6] = b.z; mk[i][7] = b.w;
          }
        }
        if (want_prev) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (rbase[i] < 0) continue;
            const float* op = reinterpret_cast<const float*>(p.out) + rbase[i] + ch * 32 + c0;
            float4 a = sg_ld4(op), b = sg_ld4(op + 4);
            prev[i][0] = a.x; prev[i][1] = a.y; prev[i][2] = a.z; prev[i][3] = a.w; prev[i][4] = b.x; prev[i][5] = b.y; prev[i][6] = b.z; prev[i][7] = b.w;
          }
        }
        uint32_t v[32];
        tmem_ld32(taddr + ch * 32, v);
        {
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          if (peers) {
            // sum over the tile's units in unit order, this unit's own accumulators at its own position
            float acc[32];
            const long long unit_f4 = (long long)nchunks * 8 * 128;
            for (int sp = 0; sp < p.split; ++sp) {
              float t[32];
              if (sp == u.si) {
#pragma unroll
                for (int j = 0; j < 32; ++j) t[j] = f[j];
              } else {
                const float4* q = peers + sp * unit_f4 + (long long)ch * 8 * 128 + row;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  float4 a = __ldcg(q + j * 128);
                  t[4 * j] = a.x; t[4 * j + 1] = a.y; t[4 * j + 2] = a.z; t[4 * j + 3] = a.w;
                }
              }
              if (sp == 0) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = t[j];
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] += t[j];
              }
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = acc[j];
          }
          if (p.bias) {
            const float* bp = p.bias + col_t * p.BN + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 b = __ldg(reinterpret_cast<const float4*>(bp + j));
              f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
            }
          }
          if (p.r1_x) {
            const float* wp = p.r1_w + col_t * p.BN + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 w4 = __ldg(reinterpret_cast<const float4*>(wp + j));
              f[j] = fmaf(r1, w4.x, f[j]); f[j + 1] = fmaf(r1, w4.y, f[j + 1]); f[j + 2] = fmaf(r1, w4.z, f[j + 2]); f[j + 3] = fmaf(r1, w4.w, f[j + 3]);
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = f[j];
          __syncwarp();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (rbase[i] < 0) continue;
          const float* sp = stg + (tr0 + 8 * i) * 33 + c0;
          float f[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = sp[j];
          const long long off = rbase[i] + ch * 32 + c0;
          if (p.mask) {
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = mk[i][j] > 0.f ? f[j] : 0.f;
          }
          if (p.out_dt == SG_F32) {
            float* op = reinterpret_cast<float*>(p.out) + off;
            if (want_prev) {
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] += prev[i][j];
            }
            sg_st4(op, make_float4(f[0], f[1], f[2], f[3]));
            sg_st4(op + 4, make_float4(f[4], f[5], f[6], f[7]));
          } else {
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + off;
            uint4 pk;
            pk.x = pack2(f[0], f[1]); pk.y = pack2(f[2], f[3]); pk.z = pack2(f[4], f[5]); pk.w = pack2(f[6], f[7]);
            *reinterpret_cast<uint4*>(op) = pk;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_tempty + 8 * as);
      as ^= 1;
      if (as == 0) aph ^= 1;
      if (peers) {
        // the last unit to leave the tile re-arms its counters for the next launch (every peer has read the partials it needs)
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (threadIdx.x == 64) {
          unsigned int* cn = p.cnt + 2 * u.tail_tile;
          if (atomicAdd(cn + 1, 1u) == (unsigned int)p.split - 1u) { cn[0] = 0u; cn[1] = 0u; __threadfence(); }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TC_TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------
// filter-gradient kernel
// ---------------------------------------------------------------------------------------------------
struct alignas(64) TcWgradParams {
  CUtensorMap map_dy;           // phase view of dy selected by (out_py, out_px, out_sy, out_sx)
  CUtensorMap map_in[4];        // sampling-phase views of the layer input
  int tap_view[SG_MAX_TAPS], tap_oy[SG_MAX_TAPS], tap_ox[SG_MAX_TAPS];
  long long tap_w_off[SG_MAX_TAPS];
  long long w_ci_stride, w_co_stride;
  int ntaps, c_in, c_out;
  int TW, TH, TN, tiles_x, tiles_y, tiles_n;      // pixel boxes; PR = TW*TH*TN pixels per k-block
  int co_tiles, ci_tiles, BN, splits, ptiles_per_split;
  int a_chunks, b_chunks, stages;
  uint32_t chunk_bytes, stage_stride;
  float* dw;
  unsigned int* sems;           // one semaphore / ticket per (tap, co tile, ci tile)
  float* db;                    // optional bias gradient [c_out] += column sums of dy (extra "bias units", see the kernel); db2: a second
  float* db2;                   //   bias that sees the same upstream gradient (the block's shortcut conv)
  float* bias_partial;          // [co_tiles][splits][128] partial column sums when splits > 1
  float* partial;               // det_mode 2: per-(tile, split) partial tiles [128][BN] fp32
  int det_mode;                 // how the pixel splits of a filter tile are combined (always in split order: bitwise repeatable)
                                //   0: one split, added straight into dw   1: ordered turns (<= 4 splits)
                                //   2: partial tiles in scratch, grid barrier, summation shared by all CTAs (many splits)
};

template <typename TIn>
__global__ void __launch_bounds__(TC_THREADS, 1) k_wgrad_tc(const __grid_constant__ TcWgradParams p) {
  constexpr bool kTf32 = sizeof(TIn) == 4;
  constexpr int KC = 128 / sizeof(TIn);
  constexpr int UK = 32 / sizeof(TIn);             // pixels consumed per tcgen05.mma
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[2 * TC_MAX_STAGES + 4];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t s_last;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = smem_u32(&bars[0]);
  const uint32_t bar_empty = smem_u32(&bars[TC_MAX_STAGES]);
  const uint32_t bar_tfull = smem_u32(&bars[2 * TC_MAX_STAGES]);
  const uint32_t bar_tempty = smem_u32(&bars[2 * TC_MAX_STAGES + 2]);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, 128);
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.map_dy);
    for (int v = 0; v < 4; ++v) tma_prefetch_desc(&p.map_in[v]);
  }
  if (p.db) {
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem_raw + (smem_base - smem_u32(smem_raw)) + p.stages * p.stage_stride);
    const uint32_t one = kTf32 ? 0x3F800000u : 0x3F803F80u;
    for (int i = threadIdx.x; i < p.TW * p.TH * p.TN * 32; i += TC_THREADS) ones[i] = one;
    fence_proxy_async();                                  // generic-proxy writes -> visible to the tensor core's async proxy
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_slot), TC_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  const int ptiles = p.tiles_x * p.tiles_y * p.tiles_n;
  const int units_w = p.ntaps * p.co_tiles * p.ci_tiles * p.splits;
  // Bias units (p.db != NULL): the bias gradient of the layer is the column sum of dy, i.e. dy^T . 1 -- one more
  // accumulation of the SAME A tiles against a constant all-ones B tile of 16 columns.  They are appended to the unit list
  // as (co tile, pixel split) units that load only A and issue N = 16 MMAs: the separate column-sum launch over dy goes away.
  const int units = units_w + (p.db ? p.co_tiles * p.splits : 0);
  const int PR = p.TW * p.TH * p.TN;
  const uint32_t ones_addr = smem_base + p.stages * p.stage_stride;      // PR x 128 bytes of 1.0 (layout-agnostic: all equal)

  // unit -> (ci tile fastest, co tile, tap, pixel split slowest): the CTAs of one wave work on the SAME pixel range with
  // different (tap, co, ci) tiles, so every dy / input tile is fetched from HBM once and shared through L2
  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < units; u += gridDim.x) {
        const int base_units = p.ntaps * p.co_tiles * p.ci_tiles;
        const bool bias_u = u >= units_w;
        int sp, cit = 0, cot, t = 0;
        if (bias_u) {
          cot = (u - units_w) % p.co_tiles;
          sp = (u - units_w) / p.co_tiles;
        } else {
          int r = u % base_units;
          sp = u / base_units;
          cit = r % p.ci_tiles; r /= p.ci_tiles;
          cot = r % p.co_tiles;
          t = r / p.co_tiles;
        }
        int pt0 = sp * p.ptiles_per_split, pt1 = pt0 + p.ptiles_per_split;
        if (pt1 > ptiles) pt1 = ptiles;
        const CUtensorMap* mi = &p.map_in[p.tap_view[t]];
        const int nb = bias_u ? 0 : p.b_chunks;
        for (int pt = pt0; pt < pt1; ++pt) {
          int tx = pt % p.tiles_x, q = pt / p.tiles_x;
          int ty = q % p.tiles_y, tn = q / p.tiles_y;
          int x0 = tx * p.TW, y0 = ty * p.TH, n0 = tn * p.TN;
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          mbar_expect_tx(bar_full + 8 * s, (p.a_chunks + nb) * p.chunk_bytes);
          uint32_t dst = smem_base + s * p.stage_stride;
          for (int j = 0; j < p.a_chunks; ++j)
            tma_load_4d(dst + j * p.chunk_bytes, &p.map_dy, bar_full + 8 * s, cot * 128 + j * KC, x0, y0, n0);
          dst += p.a_chunks * p.chunk_bytes;
          for (int j = 0; j < nb; ++j)
            tma_load_4d(dst + j * p.chunk_bytes, mi, bar_full + 8 * s, cit * p.BN + j * KC, x0 + p.tap_ox[t], y0 + p.tap_oy[t], n0);
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc_w = make_idesc(kTf32, true, true, 128, p.BN), idesc_b = make_idesc(kTf32, true, true, 128, 16);
    int s = 0, as = 0;
    uint32_t ph = 0, aph = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const bool bias_u = u >= units_w;
      const uint32_t idesc = bias_u ? idesc_b : idesc_w;
      int sp = bias_u ? (u - units_w) / p.co_tiles : u / (p.ntaps * p.co_tiles * p.ci_tiles);
      int pt0 = sp * p.ptiles_per_split, pt1 = pt0 + p.ptiles_per_split;
      if (pt1 > ptiles) pt1 = ptiles;
      mbar_wait(bar_tempty + 8 * as, aph ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)as * 256u;
      for (int pt = pt0; pt < pt1; ++pt) {
        mbar_wait(bar_full + 8 * s, ph);
        tc_fence_after();
        if (lane == 0) {
          uint32_t a_addr = smem_base + s * p.stage_stride;
          uint32_t b_addr = a_addr + p.a_chunks * p.chunk_bytes;
          // MN-major, 128B swizzle: LBO = distance between 128-byte channel chunks, SBO = distance between swizzle atoms
          // along the pixel (K) axis: 8 pixel rows = 1024 B with 16-byte atoms (bf16); tf32 MN-major operands must use the
          // 32-byte-atom variant of the 128B swizzle (TMA: SWIZZLE_128B_ATOM_32B), whose pattern repeats every 4 rows = 512 B
          uint64_t da = make_smem_desc(a_addr, p.chunk_bytes, kTf32 ? 512 : 1024, kTf32 ? 1 : 2);
          uint64_t db = make_smem_desc(bias_u ? ones_addr : b_addr, p.chunk_bytes, kTf32 ? 512 : 1024, kTf32 ? 1 : 2);
          const int ksteps = PR / UK;
          const uint32_t kadv = (UK * 128) >> 4;
          for (int k = 0; k < ksteps; ++k)
            umma<kTf32>(d_tmem, da + (uint64_t)(k * kadv), db + (uint64_t)(k * kadv), idesc, (pt != pt0 || k != 0) ? 1u : 0u);
          umma_commit(bar_empty + 8 * s);
          if (pt == pt1 - 1) umma_commit(bar_tfull + 8 * as);
        }
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1; }
      }
      as ^= 1;
      if (as == 0) aph ^= 1;
    }
  } else {
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;           // accumulator row = output channel inside the co tile
    int as = 0;
    uint32_t aph = 0;
    const int base_units = p.ntaps * p.co_tiles * p.ci_tiles;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      if (u >= units_w) {
        // ---- bias unit: column 0 of the 16-column accumulator = sum over this split's pixels of dy[:, co] ----
        const int cot_b = (u - units_w) % p.co_tiles, sp_b = (u - units_w) / p.co_tiles;
        const int co_b = cot_b * 128 + row;
        mbar_wait(bar_tfull + 8 * as, aph);
        tc_fence_after();
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)as * 256u, v);
        tc_fence_before();
        mbar_arrive(bar_tempty + 8 * as);
        const float part = __uint_as_float(v[0]);
        if (p.splits == 1) {
          if (co_b < p.c_out) {
            atomicAdd(p.db + co_b, part);
            if (p.db2) atomicAdd(p.db2 + co_b, part);
          }
        } else {
          // partial sums of the splits in scratch, added in split order by the split that arrives last (common.cuh scheme B)
          float* slots = p.bias_partial + (long long)cot_b * p.splits * 128;
          __stcg(slots + sp_b * 128 + row, part);
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (threadIdx.x == 64) {
            __threadfence();
            unsigned int tk = atomicAdd(p.sems + base_units + 2 + cot_b, 1u);
            s_last = (tk == (unsigned int)p.splits - 1) ? 1u : 0u;
            if (s_last) { p.sems[base_units + 2 + cot_b] = 0u; __threadfence(); }
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (s_last && co_b < p.c_out) {
            float tot = 0.f;
            for (int s2 = 0; s2 < p.splits; ++s2) tot += __ldcg(slots + s2 * 128 + row);
            atomicAdd(p.db + co_b, tot);
            if (p.db2) atomicAdd(p.db2 + co_b, tot);
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        as ^= 1;
        if (as == 0) aph ^= 1;
        continue;
      }
      const int tile = u % base_units, sp = u / base_units;
      int r = tile;
      int cit = r % p.ci_tiles; r /= p.ci_tiles;
      int cot = r % p.co_tiles;
      int t = r / p.co_tiles;
      int co = cot * 128 + row;
      bool valid = co < p.c_out;
      float* wbase = p.dw + p.tap_w_off[t] + (long long)co * p.w_co_stride;
      mbar_wait(bar_tfull + 8 * as, aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)as * 256u;
      if (p.det_mode == 2) {
        // Many pixel splits: every split stores its partial tile in its own scratch slot (one 128-byte line per lane and
        // chunk); after the unit loop the whole grid meets at a barrier and ALL CTAs share the ordered summation (below).
        // slot layout [BN / 4 column groups][128 rows] of float4: one store instruction of a warp (fixed column group, 32
        // consecutive rows) writes 512 contiguous bytes
        float4* slot = reinterpret_cast<float4*>(p.partial + ((long long)tile * p.splits + sp) * (128 * p.BN)) + row;
        for (int ch = 0; ch < p.BN / 32; ++ch) {
          uint32_t v[32];
          tmem_ld32(taddr + ch * 32, v);
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            __stcg(slot + (long long)(ch * 8 + j / 4) * 128,
                   make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])));
        }
        tc_fence_before();
        mbar_arrive(bar_tempty + 8 * as);
      } else {
        // Ordered turns (common.cuh, scheme A): the few pixel splits of one filter tile add their partial tiles in split
        // order.  Unit (tile, sp) only waits on unit (tile, sp - 1), which has a lower unit index: it was taken earlier by
        // its CTA (static round-robin, every CTA walks its units in increasing order), so the wait always ends.
        if (p.det_mode == 1) {
          if (threadIdx.x == 64) sg_turn_wait(p.sems + tile, (unsigned int)sp);
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        for (int ch = 0; ch < p.BN / 32; ++ch) {
          uint32_t v[32];
          tmem_ld32(taddr + ch * 32, v);
          if (valid) {
            int ci0 = cit * p.BN + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              int ci = ci0 + j;
              if (ci < p.c_in) atomicAdd(wbase + (long long)ci * p.w_ci_stride, __uint_as_float(v[j]));
            }
          }
        }
        if (p.det_mode == 1) {
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (threadIdx.x == 64) sg_turn_pass(p.sems + tile, (unsigned int)sp, (unsigned int)p.splits);
        }
        tc_fence_before();
        mbar_arrive(bar_tempty + 8 * as);
      }
      as ^= 1;
      if (as == 0) aph ^= 1;
    }
    if (p.det_mode == 2) {
      // Grid-wide phase 2 (all CTAs are co-resident: the grid never exceeds the SM count and a CTA owns its SM): once every
      // CTA has stored its partial tiles, the epilogue threads of the WHOLE grid add the splits of every filter-tile element
      // in split order -- a fixed order of additions, shared by ~19 000 threads instead of one chain per tile.
      unsigned int* gbar = p.sems + base_units;              // [0]: arrivals before phase 2, [1]: departures after it
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (threadIdx.x == 64) {
        __threadfence();
        atomicAdd(gbar, 1u);
        unsigned int v, spins = 0;
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(gbar) : "memory");
          if (v >= gridDim.x) break;
          if (++spins > (1u << 28)) __trap();
          __nanosleep(64);
        } while (true);
        __threadfence();
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const int q4 = p.BN / 4;                               // float4 column groups per accumulator row
      const long long items = (long long)base_units * q4 * 128;
      const long long tile_v4 = (long long)32 * p.BN;        // float4 per partial tile
      for (long long it = (long long)blockIdx.x * 128 + (threadIdx.x - 64); it < items; it += (long long)gridDim.x * 128) {
        const int r_ = (int)(it % 128);                      // row fastest: a warp reads / writes 32 consecutive rows
        const long long rr = it / 128;
        const int jj = (int)(rr % q4), tile = (int)(rr / q4);
        int q = tile;
        const int cit = q % p.ci_tiles; q /= p.ci_tiles;
        const int cot = q % p.co_tiles;
        const int t = q / p.co_tiles;
        const int co = cot * 128 + r_, ci = cit * p.BN + 4 * jj;
        if (co >= p.c_out || ci >= p.c_in) continue;
        const float4* src = reinterpret_cast<const float4*>(p.partial) + (long long)tile * p.splits * tile_v4 + (long long)jj * 128 + r_;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int s2 = 0; s2 < p.splits; ++s2) {
          float4 v = __ldcg(src + (long long)s2 * tile_v4);
          a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        float* wp = p.dw + p.tap_w_off[t] + (long long)co * p.w_co_stride + (long long)ci * p.w_ci_stride;
        atomicAdd(wp, a.x);                                  // exclusive owner of these four elements: RED = fire and forget
        if (ci + 1 < p.c_in) atomicAdd(wp + p.w_ci_stride, a.y);
        if (ci + 2 < p.c_in) atomicAdd(wp + 2 * p.w_ci_stride, a.z);
        if (ci + 3 < p.c_in) atomicAdd(wp + 3 * p.w_ci_stride, a.w);
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (threadIdx.x == 64) {                               // the last CTA to leave clears the barrier words for the next launch
        unsigned int left = atomicAdd(gbar + 1, 1u);
        if (left == gridDim.x - 1) { gbar[0] = 0u; gbar[1] = 0u; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TC_TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------
// weight packing: w_packed[co][t*c_in + ci] = cast(w_master[tap_w_off[t] + ci*s_ci + co*s_co])
// ---------------------------------------------------------------------------------------------------
template <typename TO>
__global__ void k_pack_weights(sg_conv_desc d, const float* __restrict__ w, TO* __restrict__ out) {
  const long long ktot = (long long)d.ntaps * d.c_in;
  const long long total = ktot * d.c_out;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int co = (int)(i / ktot);
    int k = (int)(i % ktot);
    int t = k / d.c_in, ci = k % d.c_in;
    sg_st(out + i, w[d.tap_w_off[t] + (long long)ci * d.w_ci_stride + (long long)co * d.w_co_stride]);
  }
}

// master layout with the descriptor's c_in fastest (w_ci_stride == 1, c_in % 8 == 0): 8 consecutive ci per thread,
// two float4 loads -> one 16/32-byte store
template <typename TO>
__global__ void __launch_bounds__(256) k_pack_weights_v8(sg_conv_desc d, const float* __restrict__ w, TO* __restrict__ out) {
  const int c8 = d.c_in / 8;
  const long long total8 = (long long)d.c_out * d.ntaps * c8;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total8; i += stride) {
    int g = (int)(i % c8);
    long long r = i / c8;
    int t = (int)(r % d.ntaps);
    int co = (int)(r / d.ntaps);
    const float* src = w + d.tap_w_off[t] + (long long)co * d.w_co_stride + 8 * g;
    float4 a = sg_ld4(src), b = sg_ld4(src + 4);
    TO* dst = out + i * 8;
    sg_st4(dst, a);
    sg_st4(dst + 4, b);
  }
}

// same packing when the master layout has c_out fastest (w_co_stride == 1, i.e. HWIO forward convs): a 32 x 32
// shared-memory tile transpose per tap so that both the fp32 reads (along co) and the packed writes (along ci) are
// coalesced.  grid = (ci tiles, co tiles, taps), block = 32 x 8.
template <typename TO>
__global__ void __launch_bounds__(256) k_pack_weights_t(sg_conv_desc d, const float* __restrict__ w, TO* __restrict__ out) {
  __shared__ float tile[32][33];
  const int t = blockIdx.z;
  const int ci0 = blockIdx.x * 32, co0 = blockIdx.y * 32;
  const float* src = w + d.tap_w_off[t];
#pragma unroll
  for (int j = 0; j < 32; j += 8) {
    int ci = ci0 + threadIdx.y + j, co = co0 + threadIdx.x;
    tile[threadIdx.y + j][threadIdx.x] = (ci < d.c_in && co < d.c_out) ? src[(long long)ci * d.w_ci_stride + co] : 0.f;
  }
  __syncthreads();
  const long long ktot = (long long)d.ntaps * d.c_in;
#pragma unroll
  for (int j = 0; j < 32; j += 8) {
    int co = co0 + threadIdx.y + j, ci = ci0 + threadIdx.x;
    if (ci < d.c_in && co < d.c_out) sg_st(out + (long long)co * ktot + (long long)t * d.c_in + ci, tile[threadIdx.x][threadIdx.y + j]);
  }
}

// Several packing jobs in ONE launch (the forward filters of a whole network after an optimizer step): block b belongs to
// the job whose tile range contains it.  kind 0: transposing pack of an HWIO filter (k_pack_weights_t's 32 x 32 tiles);
// kind 1: 8-wide vector copy of a filter whose master layout already has the descriptor's c_in fastest.
#define PACK_MAX_JOBS 32
struct PackJob {
  const float* src;
  void* dst;
  long long tap_stride, w_ci_stride, w_co_stride;
  int c_in, c_out, ntaps, kind, tile0, tiles_ci, tiles_co, dt;
};
struct PackJobs {
  int njobs, total_tiles;
  PackJob job[PACK_MAX_JOBS];
};
template <typename TO>
__device__ __forceinline__ void pack_tile_t(const PackJob& j, int tile, float (*smt)[33]) {
  const int tci = tile % j.tiles_ci, r = tile / j.tiles_ci;
  const int tco = r % j.tiles_co, t = r / j.tiles_co;
  const int ci0 = tci * 32, co0 = tco * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* src = j.src + (long long)t * j.tap_stride;
  TO* out = reinterpret_cast<TO*>(j.dst);
#pragma unroll
  for (int q = 0; q < 32; q += 8) {
    int ci = ci0 + ty + q, co = co0 + tx;
    smt[ty + q][tx] = (ci < j.c_in && co < j.c_out) ? src[(long long)ci * j.w_ci_stride + co] : 0.f;
  }
  __syncthreads();
  const long long ktot = (long long)j.ntaps * j.c_in;
#pragma unroll
  for (int q = 0; q < 32; q += 8) {
    int co = co0 + ty + q, ci = ci0 + tx;
    if (ci < j.c_in && co < j.c_out) sg_st(out + (long long)co * ktot + (long long)t * j.c_in + ci, smt[tx][ty + q]);
  }
}
template <typename TO>
__device__ __forceinline__ void pack_tile_v8(const PackJob& j, int tile) {
  const int c8 = j.c_in / 8;
  const long long total8 = (long long)j.c_out * j.ntaps * c8;
  const long long i = (long long)tile * 256 + threadIdx.x;
  if (i >= total8) return;
  const int g = (int)(i % c8);
  const long long r = i / c8;
  const int t = (int)(r % j.ntaps), co = (int)(r / j.ntaps);
  const float* src = j.src + (long long)t * j.tap_stride + (long long)co * j.w_co_stride + 8 * g;
  float4 a = sg_ld4(src), b = sg_ld4(src + 4);
  TO* dst = reinterpret_cast<TO*>(j.dst) + i * 8;
  sg_st4(dst, a);
  sg_st4(dst + 4, b);
}
__global__ void __launch_bounds__(256) k_pack_weights_multi(const __grid_constant__ PackJobs jobs) {
  __shared__ float smt[32][33];
  int ji = 0;
  while (ji + 1 < jobs.njobs && (int)blockIdx.x >= jobs.job[ji + 1].tile0) ++ji;
  const PackJob& j = jobs.job[ji];
  const int tile = blockIdx.x - j.tile0;
  if (j.kind == 0) {
    if (j.dt == SG_F32) pack_tile_t<float>(j, tile, smt);
    else pack_tile_t<__nv_bfloat16>(j, tile, smt);
  } else {
    if (j.dt == SG_F32) pack_tile_v8<float>(j, tile);
    else pack_tile_v8<__nv_bfloat16>(j, tile);
  }
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int get_encode(sg_ctx* ctx, PFN_encodeTiled* fn) {
  if (!ctx->encode_tiled) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    SG_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres));
    SG_REQUIRE(f != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    ctx->encode_tiled = f;
  }
  *fn = (PFN_encodeTiled)ctx->encode_tiled;
  return SG_OK;
}

static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
static inline int posmod(int a, int b) { return a - floordiv(a, b) * b; }

// 4-D NHWC view (optionally a stride-phase view): dims {c, wv, hv, n}
static int encode_nhwc_view(PFN_encodeTiled enc, CUtensorMap* m, int dt, const void* base, int n, int h, int w, int c, int sy,
                            int sx, int py, int px, int box_c, int box_w, int box_h, int box_n,
                            CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  size_t e = dt == SG_F32 ? 4 : 2;
  int hv = (h - py + sy - 1) / sy, wv = (w - px + sx - 1) / sx;
  if (hv < 1) hv = 1;
  if (wv < 1) wv = 1;
  cuuint64_t gdim[4] = {(cuuint64_t)c, (cuuint64_t)wv, (cuuint64_t)hv, (cuuint64_t)n};
  cuuint64_t gstr[3] = {(cuuint64_t)sx * c * e, (cuuint64_t)sy * w * c * e, (cuuint64_t)h * w * c * e};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_n};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const char* addr = (const char*)base + ((size_t)py * w + px) * c * e;
  CUresult r = enc(m, dt == SG_F32 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)addr, gdim,
                   gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    sg_set_error("cuTensorMapEncodeTiled(4d) failed: %d (dims %d,%d,%d,%d box %d,%d,%d,%d)", (int)r, c, wv, hv, n, box_c, box_w,
                 box_h, box_n);
    return SG_ERR_CUDA;
  }
  return SG_OK;
}

static int encode_2d(PFN_encodeTiled enc, CUtensorMap* m, int dt, const void* base, long long inner, long long outer, int box_in,
                     int box_out) {
  size_t e = dt == SG_F32 ? 4 : 2;
  cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t gstr[1] = {(cuuint64_t)inner * e};
  cuuint32_t box[2] = {(cuuint32_t)box_in, (cuuint32_t)box_out};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, dt == SG_F32 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)base, gdim,
                   gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    sg_set_error("cuTensorMapEncodeTiled(2d) failed: %d (dims %lld,%lld box %d,%d)", (int)r, inner, outer, box_in, box_out);
    return SG_ERR_CUDA;
  }
  return SG_OK;
}

// choose a pixel box TW x TH x TN (<= max_rows pixels, product a multiple of `mult`) minimising the padded MMA
// work.  Boxes may overhang the image: the overhang is TMA zero-fill on load and predicated off on store.
static void choose_box(int gw, int gh, int n, int max_rows, int mult, int* TW, int* TH, int* TN) {
  struct Key { int gw, gh, n, mr, mu, tw, th, tn; };
  static thread_local Key cache[64];
  static thread_local int cache_n = 0;
  for (int i = 0; i < cache_n; ++i)
    if (cache[i].gw == gw && cache[i].gh == gh && cache[i].n == n && cache[i].mr == max_rows && cache[i].mu == mult) {
      *TW = cache[i].tw; *TH = cache[i].th; *TN = cache[i].tn;
      return;
    }
  long long best = -1;
  int bw = mult, bh = 1, bn = 1;
  int last_tw = -1;
  for (int kx = 1; kx <= gw; ++kx) {
    int tw = (gw + kx - 1) / kx;
    if (tw == last_tw) continue;
    last_tw = tw;
    if (tw > max_rows || tw > 256) continue;
    int last_th = -1;
    for (int ky = 1; ky <= gh; ++ky) {
      int th = (gh + ky - 1) / ky;
      if (th == last_th) continue;
      last_th = th;
      if ((long long)tw * th > max_rows) continue;
      // a box is any rectangle in (x, y, image) space: several images may share a box even when it covers only
      // part of each image (e.g. 20 x 2 rows x 3 images = 120 of 128 accumulator rows for an 8 x 20 map)
      int tn = max_rows / (tw * th);
      if (tn > n) tn = n;
      if (tn < 1) tn = 1;
      int tw2 = tw, tn2 = tn;
      bool ok = false;
      for (; tn2 >= 1; --tn2)
        if (((long long)tw2 * th * tn2) % mult == 0) { ok = true; break; }
      if (!ok) {
        tn2 = 1;
        for (tw2 = tw; (long long)tw2 * th <= max_rows && tw2 <= 256; ++tw2)
          if (((long long)tw2 * th) % mult == 0) { ok = true; break; }
      }
      if (!ok) continue;
      long long pr = (long long)tw2 * th * tn2;
      long long tiles = (long long)((gw + tw2 - 1) / tw2) * ((gh + th - 1) / th) * ((n + tn2 - 1) / tn2);
      // forward kernel (mult == 1): every tile costs one full M=128 accumulation, so minimise the tile count;
      // filter-gradient kernel: pixels are the reduction dim, so minimise the padded pixel count
      long long cost = (mult == 1) ? tiles * 1024 - pr : tiles * pr + tiles;
      if (best < 0 || cost < best) { best = cost; bw = tw2; bh = th; bn = tn2; }
    }
  }
  if (cache_n < 64) { Key k = {gw, gh, n, max_rows, mult, bw, bh, bn}; cache[cache_n++] = k; }
  *TW = bw; *TH = bh; *TN = bn;
}

// pixel splits of the filter gradient: static round-robin over #SMs persistent CTAs costs ceil(units / #SMs) unit-times, so
// pick the split count whose last wave is fullest (e.g. 72 base units: 4 splits = 288 units = 1.95 waves, not 5 splits = 2.43)
static int wgrad_choose_splits(int ptiles, long long base_units, int co_tiles, int num_sms) {
  int max_splits = sg_div_up(ptiles, 8);           // at least 8 k-blocks per unit
  if (max_splits > 32) max_splits = 32;
  if (base_units + 2 + co_tiles > SG_DET_TICKETS) max_splits = 1;  // no turn semaphores for that many filter tiles
  int splits = 1;
  double best_eff = -1.0;
  for (int sp = 1; sp <= max_splits; ++sp) {
    int pps = sg_div_up(ptiles, sp);
    int eff_sp = sg_div_up(ptiles, pps);
    if (eff_sp != sp) continue;
    long long units_sp = base_units * sp;
    long long waves = (units_sp + num_sms - 1) / num_sms;
    // work per CTA in k-blocks: waves * pps (plus one epilogue per unit, ~ 4 k-blocks worth)
    double cost = (double)waves * (pps + 4.0);
    double eff = 1.0 / cost;
    if (eff > best_eff * 1.02) { best_eff = eff; splits = sp; }
  }
  return splits;
}

static int tc_check(const sg_conv_desc* d, const char* who) {
  SG_REQUIRE(d != nullptr, "%s: desc is NULL", who);
  int kc = d->in_dt == SG_F32 ? 32 : 64;
  SG_REQUIRE(d->in_dt == SG_F32 || d->in_dt == SG_BF16, "%s: bad in_dt", who);
  SG_REQUIRE(d->c_in % kc == 0, "%s: c_in=%d must be a multiple of %d for the tensor-core path", who, d->c_in, kc);
  SG_REQUIRE(d->c_out % 32 == 0, "%s: c_out=%d must be a multiple of 32 for the tensor-core path", who, d->c_out);
  SG_REQUIRE(d->ntaps >= 1 && d->ntaps <= SG_MAX_TAPS, "%s: bad ntaps", who);
  SG_REQUIRE(d->in_sy >= 1 && d->in_sy <= 2 && d->in_sx >= 1 && d->in_sx <= 2, "%s: input sampling stride must be 1 or 2", who);
  SG_REQUIRE(d->n > 0 && d->grid_h > 0 && d->grid_w > 0, "%s: empty problem", who);
  return SG_OK;
}

extern "C" {

int sg_conv_tc_supported(const sg_conv_desc* d) {
  if (!d) return 0;
  int kc = d->in_dt == SG_F32 ? 32 : 64;
  return (d->c_in % kc == 0) && (d->c_out % 32 == 0) && d->in_sy <= 2 && d->in_sx <= 2 && d->ntaps >= 1 &&
         d->ntaps <= SG_MAX_TAPS && d->n > 0;
}

size_t sg_conv_packed_weight_elems(const sg_conv_desc* d) {
  return d ? (size_t)d->c_out * d->ntaps * d->c_in : 0;
}

int sg_conv_pack_weights(sg_ctx* ctx, const sg_conv_desc* d, const float* w_master, void* w_packed) {
  SG_REQUIRE(ctx && d && w_master && w_packed, "sg_conv_pack_weights: NULL");
  long long total = (long long)d->c_out * d->ntaps * d->c_in;
  if (total == 0) return SG_OK;
  if (d->w_co_stride == 1 && d->w_ci_stride != 1 && d->c_out >= 32) {
    dim3 grid(sg_div_up(d->c_in, 32), sg_div_up(d->c_out, 32), d->ntaps), block(32, 8);
    SG_DISPATCH_DT(d->in_dt, TO, sg_launch(ctx, k_pack_weights_t<TO>, grid, block, 0, *d, w_master, (TO*)w_packed));
  } else if (d->w_ci_stride == 1 && d->c_in % 8 == 0 && d->w_co_stride % 4 == 0 && ((uintptr_t)w_master & 15) == 0) {
    bool taps_ok = true;
    for (int t = 0; t < d->ntaps; ++t) taps_ok = taps_ok && (d->tap_w_off[t] % 4 == 0);
    long long need = (total / 8 + 255) / 256, cap = (long long)ctx->num_sms * 8;
    int grid = (int)(need < cap ? need : cap);
    if (taps_ok) {
      SG_DISPATCH_DT(d->in_dt, TO, sg_launch(ctx, k_pack_weights_v8<TO>, grid, 256, 0, *d, w_master, (TO*)w_packed));
    } else {
      SG_DISPATCH_DT(d->in_dt, TO, sg_launch(ctx, k_pack_weights<TO>, grid, 256, 0, *d, w_master, (TO*)w_packed));
    }
  } else {
    long long need = (total + 255) / 256, cap = (long long)ctx->num_sms * 8;
    int grid = (int)(need < cap ? need : cap);
    SG_DISPATCH_DT(d->in_dt, TO, sg_launch(ctx, k_pack_weights<TO>, grid, 256, 0, *d, w_master, (TO*)w_packed));
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

/* 1 when sg_conv_pack_weights_multi can take this filter (regular taps t * c_in * c_out; one of the two vectorisable layouts) */
int sg_conv_pack_multi_supported(const sg_conv_desc* d, const float* w_master) {
  if (!d) return 0;
  const long long ts = (long long)d->c_in * d->c_out;
  for (int t = 0; t < d->ntaps; ++t)
    if (d->tap_w_off[t] != (long long)t * ts) return 0;
  if (d->w_co_stride == 1 && d->w_ci_stride != 1 && d->c_out >= 32) return 1;
  if (d->w_ci_stride == 1 && d->c_in % 8 == 0 && d->w_co_stride % 4 == 0 && ((uintptr_t)w_master & 15) == 0 && ts % 4 == 0) return 1;
  return 0;
}

/* njobs (<= 32) packing jobs in one launch: descs / w_master / w_packed are HOST arrays of length njobs */
int sg_conv_pack_weights_multi(sg_ctx* ctx, int njobs, const sg_conv_desc* const* descs, const float* const* w_master, void* const* w_packed) {
  SG_REQUIRE(ctx && descs && w_master && w_packed && njobs >= 1 && njobs <= PACK_MAX_JOBS, "sg_conv_pack_weights_multi: bad args");
  static_assert(sizeof(PackJobs) < 4000, "kernel parameter block too large");
  PackJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  jobs.njobs = njobs;
  int tile = 0;
  for (int i = 0; i < njobs; ++i) {
    const sg_conv_desc* d = descs[i];
    SG_REQUIRE(d && w_master[i] && w_packed[i] && sg_conv_pack_multi_supported(d, w_master[i]), "sg_conv_pack_weights_multi: job %d not supported", i);
    PackJob& j = jobs.job[i];
    j.src = w_master[i]; j.dst = w_packed[i];
    j.tap_stride = (long long)d->c_in * d->c_out; j.w_ci_stride = d->w_ci_stride; j.w_co_stride = d->w_co_stride;
    j.c_in = d->c_in; j.c_out = d->c_out; j.ntaps = d->ntaps; j.dt = d->in_dt;
    j.tile0 = tile;
    if (d->w_co_stride == 1 && d->w_ci_stride != 1 && d->c_out >= 32) {
      j.kind = 0;
      j.tiles_ci = sg_div_up(d->c_in, 32); j.tiles_co = sg_div_up(d->c_out, 32);
      tile += j.tiles_ci * j.tiles_co * d->ntaps;
    } else {
      j.kind = 1;
      long long total8 = (long long)d->c_out * d->ntaps * (d->c_in / 8);
      tile += (int)((total8 + 255) / 256);
    }
  }
  jobs.total_tiles = tile;
  if (tile == 0) return SG_OK;
  sg_launch(ctx, k_pack_weights_multi, tile, 256, 0, jobs);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

static int encode_3d(PFN_encodeTiled enc, CUtensorMap* m, const void* base, long long d0, long long d1, long long d2, long long s1,
                     long long s2, int b0, int b1) {
  cuuint64_t gdim[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t gstr[2] = {(cuuint64_t)s1 * 2, (cuuint64_t)s2 * 2};          // bf16
  cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    sg_set_error("cuTensorMapEncodeTiled(3d) failed: %d (dims %lld,%lld,%lld strides %lld,%lld box %d,%d)", (int)r, d0, d1, d2, s1, s2, b0, b1);
    return SG_ERR_CUDA;
  }
  return SG_OK;
}

// 0 = not possible; 1 = master is K-major for this role (w_ci_stride == 1); 2 = N-major (w_co_stride == 1)
static int direct_mode(const sg_conv_desc* d) {
  if (!d || d->in_dt != SG_BF16) return 0;
  if (d->c_in % 64 || d->c_out % 32) return 0;
  const long long ts = (long long)d->c_in * d->c_out;
  for (int t = 0; t < d->ntaps; ++t)
    if (d->tap_w_off[t] < 0 || d->tap_w_off[t] % ts) return 0;
  if (d->w_ci_stride == 1 && d->w_co_stride == d->c_in) return 1;
  if (d->w_co_stride == 1 && d->w_ci_stride == d->c_out && d->c_out % 64 == 0) return 2;
  return 0;
}

// Cost (in tile-times of the given N tile) of `tiles` output tiles on `sms` persistent CTAs, and the tail split that achieves it:
// whole waves run unsplit; the tiles of the last, partial wave are cut into `split` k-ranges each (<= 8, >= 4 k-blocks per range,
// partials within the workspace).  A split wave costs ceil(rem * split / sms) / split tile-times plus the exchange: the rendezvous
// and one tile of fp32 partials written and read through L2, ~10 us measured (tools/trace_step.py), against ~0.45 us per k-block of
// a 128 x 256 tile -- i.e. ~22 k-blocks' worth, which is why short-k launches (R's deep layers, the G phases) stay unsplit.
static double tc_split_plan(long long tiles, int sms, int nkb, int bn, int enabled, int* split_out) {
  const long long full = tiles / sms, rem = tiles % sms;
  *split_out = 1;
  if (rem == 0) return (double)full;
  double best = (double)full + 1.0;
  if (!enabled) return best;
  const double exchange = 22.0 * (256.0 / (double)bn) / (double)nkb;
  for (int s = 2; s <= 8; ++s) {
    if (nkb / s < 4) break;
    if ((long long)rem * s * 128 * bn * 4 > (long long)SG_DET_SCRATCH_BYTES) break;
    if (2 * rem > SG_DET_TICKETS) break;
    const long long waves = (rem * s + sms - 1) / sms;
    const double cost = (double)full + (double)waves / s + exchange;
    if (cost < best * 0.97) { best = cost; *split_out = s; }
  }
  return best;
}

static int conv_fwd_tc_impl(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed, int b_mode, const float* bias,
                            const void* mask, void* out, const sg_conv_desc* d2 = nullptr, const void* in2 = nullptr,
                            const void* w_packed2 = nullptr, const float* r1_x = nullptr, const float* r1_w = nullptr,
                            const sg_conv_desc* const* phases = nullptr, int nphase = 1) {
  SG_REQUIRE(ctx && in && w_packed && out, "sg_conv_fwd_tc: NULL");
  int rc = tc_check(d, "sg_conv_fwd_tc");
  if (rc != SG_OK) return rc;
  SG_REQUIRE(!d->accumulate || d->out_dt == SG_F32, "sg_conv_fwd_tc: accumulate needs an fp32 output");
  SG_REQUIRE(((uintptr_t)in & 15) == 0 && ((uintptr_t)w_packed & 15) == 0 && ((uintptr_t)out & 15) == 0 &&
                 ((uintptr_t)bias & 15) == 0 && ((uintptr_t)mask & 15) == 0,
             "sg_conv_fwd_tc: pointers must be 16-byte aligned");
  PFN_encodeTiled enc;
  rc = get_encode(ctx, &enc);
  if (rc != SG_OK) return rc;

  static_assert(sizeof(TcFwdParams) < 4000, "kernel parameter block too large");
  TcFwdParams p;
  memset(&p, 0, sizeof(p));
  const int es = d->in_dt == SG_F32 ? 4 : 2;
  const int KC = 128 / es;
  p.ntaps = d->ntaps; p.c_in = d->c_in; p.c_out = d->c_out; p.n = d->n; p.grid_h = d->grid_h; p.grid_w = d->grid_w;
  p.out_h = d->out_h; p.out_w = d->out_w; p.out_sy = d->out_sy; p.out_sx = d->out_sx; p.out_py = d->out_py; p.out_px = d->out_px;
  p.relu = d->relu; p.accumulate = d->accumulate; p.out_dt = d->out_dt; p.mask_dt = d->mask_dt;
  p.bias = bias; p.mask = mask; p.out = out;
  if (r1_x) {
    SG_REQUIRE(r1_w && d->out_sy == 1 && d->out_sx == 1 && d->out_py == 0 && d->out_px == 0 && ((uintptr_t)r1_w & 15) == 0,
               "sg_conv_fwd_tc_rank1: needs a unit-stride output and a 16-byte aligned weight vector");
    p.r1_x = r1_x; p.r1_w = r1_w;
  }
  choose_box(d->grid_w, d->grid_h, d->n, 128, 1, &p.TW, &p.TH, &p.TN);
  p.tiles_x = sg_div_up(d->grid_w, p.TW); p.tiles_y = sg_div_up(d->grid_h, p.TH); p.tiles_n = sg_div_up(d->n, p.TN);
  const int nkb_total = d->ntaps * (d->c_in / KC) + (d2 ? d2->c_in / KC : 0);
  int best_split = 1;
  {
    // N tile and tail split.  With a static persistent schedule a launch costs ceil(tiles / #SMs) tile-times, so a launch whose
    // last wave is mostly empty (D.B4: 40 pixel tiles x 4 = 160 tiles of 256 columns on 148 SMs = 2 waves for 1.08 waves of work)
    // runs at half speed.  Two remedies, costed together: a narrower N tile (relative tile times from tools/bench_conv.py on
    // B200: the main loop is operand-load bound, a 128-column tile costs ~0.85 of a 256-column one), and splitting the k-range of
    // the tiles of the last, partial wave over `split` CTAs each (tc_split_plan).
    const int cand[4] = {256, 128, 64, 32};
    const double rel[4] = {1.0, 0.85, 0.75, 0.7};
    const long long m_tiles = (long long)p.tiles_x * p.tiles_y * p.tiles_n;
    double best = -1.0;
    p.BN = 32;
    for (int i = 0; i < 4; ++i) {
      if (d->c_out % cand[i]) continue;
      if (b_mode == 2 && cand[i] < 64) continue;
      long long tiles = m_tiles * (d->c_out / cand[i]) * nphase;
      int split = 1;
      double cost = tc_split_plan(tiles, ctx->num_sms, nkb_total, cand[i], ctx->conv_split_tail && nphase == 1, &split) * rel[i];
      if (best < 0 || cost < best * 0.97) { best = cost; p.BN = cand[i]; best_split = split; }
    }
  }
  p.tiles_col = d->c_out / p.BN;
  p.kc_per_tap = d->c_in / KC;
  const int PR = p.TW * p.TH * p.TN;
  p.a_bytes = (uint32_t)PR * 128u;
  p.b_bytes = (uint32_t)p.BN * 128u;
  p.a_stage_stride = 128u * 128u;                  // always reserve a full 128-row tile (1024-byte aligned)
  p.b_stage_stride = (uint32_t)p.BN * 128u;
  int stages = (int)((204u * 1024u) / (p.a_stage_stride + p.b_stage_stride));
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  SG_REQUIRE(stages >= 2, "sg_conv_fwd_tc: not enough shared memory for 2 stages");
  p.stages = stages;

  bool used[4] = {false, false, false, false};
  // tap tables: one phase = the descriptor's own taps; several phases = their taps back to back
  long long tap_w_off_all[SG_MAX_TAPS];
  {
    int nt = 0;
    p.nphase = nphase;
    for (int ph = 0; ph < nphase; ++ph) {
      const sg_conv_desc* dp = phases ? phases[ph] : d;
      p.ph_tap0[ph] = nt; p.ph_ntaps[ph] = dp->ntaps; p.ph_py[ph] = dp->out_py; p.ph_px[ph] = dp->out_px;
      for (int t = 0; t < dp->ntaps; ++t, ++nt) {
        SG_REQUIRE(nt < SG_MAX_TAPS, "sg_conv_fwd_tc_phases: more than %d taps in total", SG_MAX_TAPS);
        int py = posmod(dp->tap_dy[t], dp->in_sy), px = posmod(dp->tap_dx[t], dp->in_sx);
        int v = py * 2 + px;
        p.tap_view[nt] = v;
        p.tap_oy[nt] = floordiv(dp->tap_dy[t], dp->in_sy);
        p.tap_ox[nt] = floordiv(dp->tap_dx[t], dp->in_sx);
        tap_w_off_all[nt] = dp->tap_w_off[t];
        used[v] = true;
      }
    }
    p.ntaps = nt;
  }
  int first_used = -1;
  for (int v = 0; v < 4; ++v) {
    if (!used[v]) continue;
    if (first_used < 0) first_used = v;
    rc = encode_nhwc_view(enc, &p.map_a[v], d->in_dt, in, d->n, d->in_h, d->in_w, d->c_in, d->in_sy, d->in_sx, v / 2, v % 2, KC,
                          p.TW, p.TH, p.TN);
    if (rc != SG_OK) return rc;
  }
  for (int v = 0; v < 4; ++v)
    if (!used[v]) p.map_a[v] = p.map_a[first_used];
  if (d2) {      // second operand: a 1x1, stride-1 conv on the same pixel grid and output channels, packed K-major weights
    SG_REQUIRE(in2 && w_packed2 && b_mode == 0, "sg_conv_fwd_tc_dual: NULL second operand / needs packed weights");
    SG_REQUIRE(d2->ntaps == 1 && d2->tap_dy[0] == 0 && d2->tap_dx[0] == 0 && d2->in_sy == 1 && d2->in_sx == 1,
               "sg_conv_fwd_tc_dual: the second conv must be 1x1, stride 1");
    SG_REQUIRE(d2->n == d->n && d2->grid_h == d->grid_h && d2->grid_w == d->grid_w && d2->c_out == d->c_out && d2->in_dt == d->in_dt &&
                   d2->in_h == d->grid_h && d2->in_w == d->grid_w && d2->c_in % KC == 0,
               "sg_conv_fwd_tc_dual: the second conv must share the batch, pixel grid, output channels and operand dtype");
    SG_REQUIRE(((uintptr_t)in2 & 15) == 0 && ((uintptr_t)w_packed2 & 15) == 0, "sg_conv_fwd_tc_dual: pointers must be 16-byte aligned");
    p.kc2 = d2->c_in / KC;
    rc = encode_nhwc_view(enc, &p.map_a2, d2->in_dt, in2, d2->n, d2->in_h, d2->in_w, d2->c_in, 1, 1, 0, 0, KC, p.TW, p.TH, p.TN);
    if (rc != SG_OK) return rc;
    rc = encode_2d(enc, &p.map_b2, d2->in_dt, w_packed2, d2->c_in, d2->c_out, KC, p.BN);
    if (rc != SG_OK) return rc;
  }
  p.b_mode = b_mode;
  if (b_mode == 0) {
    rc = encode_2d(enc, &p.map_b, d->in_dt, w_packed, (long long)d->ntaps * d->c_in, d->c_out, KC, p.BN);
  } else {
    const long long ts = (long long)d->c_in * d->c_out;
    long long tmax = 0;
    for (int t = 0; t < p.ntaps; ++t) {
      p.tap_wt[t] = (int)(tap_w_off_all[t] / ts);
      if (p.tap_wt[t] > tmax) tmax = p.tap_wt[t];
    }
    if (b_mode == 1) rc = encode_3d(enc, &p.map_b, w_packed, d->c_in, d->c_out, tmax + 1, d->w_co_stride, ts, KC, p.BN);
    else rc = encode_3d(enc, &p.map_b, w_packed, d->c_out, d->c_in, tmax + 1, d->w_ci_stride, ts, 64, KC);
  }
  if (rc != SG_OK) return rc;

  p.tiles_per_phase = p.tiles_x * p.tiles_y * p.tiles_n * p.tiles_col;
  long long total_tiles = (long long)p.tiles_per_phase * nphase;
  p.split = best_split;
  p.t_full = (int)(best_split > 1 ? total_tiles / ctx->num_sms * ctx->num_sms : total_tiles);
  p.total_units = (int)(p.t_full + (total_tiles - p.t_full) * p.split);
  p.part = ctx->det_scratch;
  p.cnt = ctx->det_tickets;
  int grid = p.total_units < ctx->num_sms ? p.total_units : ctx->num_sms;
  size_t smem = (size_t)stages * (p.a_stage_stride + p.b_stage_stride) + 1024 + TC_EPI_STAGING;
  // split tiles rendezvous inside the kernel: launched cooperatively, so that all CTAs are co-resident even when a kernel of
  // another stream (rt.branch) holds part of the SMs
  const bool coop = p.split > 1;
  if (d->in_dt == SG_F32) {
    SG_CHECK_CUDA(cudaFuncSetAttribute(k_conv_tc<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SG_CHECK_CUDA(sg_launch_ex(ctx, coop, k_conv_tc<float>, grid, TC_THREADS, smem, p));
  } else {
    SG_CHECK_CUDA(cudaFuncSetAttribute(k_conv_tc<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SG_CHECK_CUDA(sg_launch_ex(ctx, coop, k_conv_tc<__nv_bfloat16>, grid, TC_THREADS, smem, p));
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_conv_fwd_tc(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed, const float* bias,
                   const void* mask, void* out) {
  return conv_fwd_tc_impl(ctx, d, in, w_packed, 0, bias, mask, out);
}

/* out = epilogue( conv(d, in, w_packed) + conv1x1(d2, in2, w_packed2) ): the ResNet block's shortcut (resnet_ops.py:109-114)
 * accumulated in TMEM as extra k-blocks of the main conv instead of a second read-modify-write pass over the output */
/* host-only: the N tile and tail split sg_conv_fwd_tc would choose for this descriptor on a device with num_sms SMs */
int sg_conv_tc_plan(const sg_conv_desc* d, int num_sms, int split_tail_enabled, int* bn_out, int* split_out, int* tiles_out) {
  SG_REQUIRE(d && num_sms > 0 && bn_out && split_out && tiles_out, "sg_conv_tc_plan: bad args");
  int rc = tc_check(d, "sg_conv_tc_plan");
  if (rc != SG_OK) return rc;
  const int KC = 128 / (d->in_dt == SG_F32 ? 4 : 2);
  int TW, TH, TN;
  choose_box(d->grid_w, d->grid_h, d->n, 128, 1, &TW, &TH, &TN);
  const long long m_tiles = (long long)sg_div_up(d->grid_w, TW) * sg_div_up(d->grid_h, TH) * sg_div_up(d->n, TN);
  const int nkb = d->ntaps * (d->c_in / KC);
  const int cand[4] = {256, 128, 64, 32};
  const double rel[4] = {1.0, 0.85, 0.75, 0.7};
  double best = -1.0;
  *bn_out = 32; *split_out = 1;
  for (int i = 0; i < 4; ++i) {
    if (d->c_out % cand[i]) continue;
    long long tiles = m_tiles * (d->c_out / cand[i]);
    int split = 1;
    double cost = tc_split_plan(tiles, num_sms, nkb, cand[i], split_tail_enabled, &split) * rel[i];
    if (best < 0 || cost < best * 0.97) { best = cost; *bn_out = cand[i]; *split_out = split; }
  }
  *tiles_out = (int)(m_tiles * (d->c_out / *bn_out));
  return SG_OK;
}

int sg_conv_fwd_tc_rank1(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed, const float* bias,
                         const void* mask, void* out, const float* r1_x, const float* r1_w) {
  SG_REQUIRE(r1_x && r1_w, "sg_conv_fwd_tc_rank1: NULL rank-1 operands");
  return conv_fwd_tc_impl(ctx, d, in, w_packed, 0, bias, mask, out, nullptr, nullptr, nullptr, r1_x, r1_w);
}

int sg_conv_fwd_tc_dual(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed, const sg_conv_desc* d2,
                        const void* in2, const void* w_packed2, const float* bias, const void* mask, void* out) {
  SG_REQUIRE(d2 != nullptr, "sg_conv_fwd_tc_dual: NULL second descriptor");
  return conv_fwd_tc_impl(ctx, d, in, w_packed, 0, bias, mask, out, d2, in2, w_packed2);
}

int sg_conv_tc_direct_supported(const sg_conv_desc* d) { return sg_conv_tc_supported(d) && direct_mode(d) != 0; }

/* same launch reading the filter IN PLACE from a bf16 mirror of the master weights (same indexing as w_master): no
 * packing pass.  Forward convs (HWIO) use it as an N-major B operand, dgrads / transposed convs as a K-major one. */
int sg_conv_fwd_tc_direct(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_mirror_bf16, const float* bias,
                          const void* mask, void* out) {
  int mode = direct_mode(d);
  SG_REQUIRE(mode != 0, "sg_conv_fwd_tc_direct: this descriptor cannot read the master filter in place");
  return conv_fwd_tc_impl(ctx, d, in, w_mirror_bf16, mode, bias, mask, out);
}

/* the output phases of a transposed conv (Conv2DTranspose forward, resnet_ops.py:57,69) as ONE launch: descs[i] are the
 * phase descriptors (ops.desc_convT_phase: same tensors and pixel grid, different taps and output offsets) */
int sg_conv_fwd_tc_phases(sg_ctx* ctx, int nphase, const sg_conv_desc* const* descs, const void* in, const void* w_mirror_bf16,
                          const float* bias, void* out) {
  SG_REQUIRE(descs && nphase >= 1 && nphase <= 4, "sg_conv_fwd_tc_phases: 1..4 phases");
  const sg_conv_desc* d = descs[0];
  int mode = direct_mode(d);
  SG_REQUIRE(mode != 0, "sg_conv_fwd_tc_phases: the phases must be able to read the master filter in place (bf16 mirror)");
  for (int i = 1; i < nphase; ++i) {
    const sg_conv_desc* e = descs[i];
    SG_REQUIRE(e && direct_mode(e) == mode && e->n == d->n && e->in_h == d->in_h && e->in_w == d->in_w && e->c_in == d->c_in &&
                   e->out_h == d->out_h && e->out_w == d->out_w && e->c_out == d->c_out && e->grid_h == d->grid_h &&
                   e->grid_w == d->grid_w && e->in_sy == d->in_sy && e->in_sx == d->in_sx && e->out_sy == d->out_sy &&
                   e->out_sx == d->out_sx && e->in_dt == d->in_dt && e->out_dt == d->out_dt && e->relu == d->relu &&
                   e->accumulate == d->accumulate && e->w_ci_stride == d->w_ci_stride && e->w_co_stride == d->w_co_stride,
               "sg_conv_fwd_tc_phases: phase %d differs from phase 0 in more than taps and output offset", i);
  }
  return conv_fwd_tc_impl(ctx, d, in, w_mirror_bf16, mode, bias, nullptr, out, nullptr, nullptr, nullptr, nullptr, nullptr, descs, nphase);
}

size_t sg_conv_wgrad_tc_workspace(const sg_conv_desc* d, int num_sms) {
  (void)d; (void)num_sms;
  return 0;      // split partials are added straight into dw in split order (turn semaphores in the context): no workspace
}

static int conv_wgrad_tc_impl(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master, float* db, float* db2);

int sg_conv_wgrad_tc(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master, void* workspace,
                     size_t workspace_bytes) {
  (void)workspace; (void)workspace_bytes;
  return conv_wgrad_tc_impl(ctx, d, in, dy, dw_master, nullptr, nullptr);
}

/* 1 when the bias units of sg_conv_wgrad_tc_bias fit into the idle CTA slots of the filter-gradient launch's last wave (then the
 * bias gradient is free); 0 when they would open an extra wave -- measured slower than a separate column-sum launch, because a
 * bias unit streams only the dy tiles (16 KB per stage in flight: latency bound) and lasts about as long as a full unit. */
int sg_conv_wgrad_tc_bias_fits(sg_ctx* ctx, const sg_conv_desc* d) {
  if (!ctx || !d || !sg_conv_tc_supported(d)) return 0;
  const int es = d->in_dt == SG_F32 ? 4 : 2;
  const int KC = 128 / es, UK = 32 / es;
  const int BN = d->c_in % 256 == 0 ? 256 : (d->c_in % 128 == 0 ? 128 : (d->c_in % 64 == 0 ? 64 : 32));
  const int ci_tiles = d->c_in / BN, co_tiles = sg_div_up(d->c_out, 128);
  int max_rows = (48 * 1024) / (128 * (128 / KC + BN / KC));
  if (max_rows > 128) max_rows = 128;
  max_rows = max_rows / UK * UK;
  int TW, TH, TN;
  choose_box(d->grid_w, d->grid_h, d->n, max_rows, UK, &TW, &TH, &TN);
  const int ptiles = sg_div_up(d->grid_w, TW) * sg_div_up(d->grid_h, TH) * sg_div_up(d->n, TN);
  const long long base_units = (long long)d->ntaps * co_tiles * ci_tiles;
  const int splits = wgrad_choose_splits(ptiles, base_units, co_tiles, ctx->num_sms);
  const long long units = base_units * splits, bias_units = (long long)co_tiles * splits;
  if (units < ctx->num_sms) return units + bias_units <= ctx->num_sms;
  const long long idle = (ctx->num_sms - units % ctx->num_sms) % ctx->num_sms;
  return bias_units <= idle;
}

/* filter gradient + bias gradient in ONE launch: db[c_out] (and db2, the bias of a shortcut conv that sees the same upstream
 * gradient; may be NULL) += column sums of dy, computed by the tensor cores as dy^T . 1 */
int sg_conv_wgrad_tc_bias(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master, float* db, float* db2) {
  SG_REQUIRE(db != nullptr, "sg_conv_wgrad_tc_bias: NULL bias gradient");
  SG_REQUIRE(d && d->out_sy == 1 && d->out_sx == 1 && d->out_py == 0 && d->out_px == 0 && d->grid_h == d->out_h && d->grid_w == d->out_w,
             "sg_conv_wgrad_tc_bias: the pixel grid must cover dy exactly once (plain Conv2D filter gradients only)");
  return conv_wgrad_tc_impl(ctx, d, in, dy, dw_master, db, db2);
}

static int conv_wgrad_tc_impl(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master, float* db, float* db2) {
  SG_REQUIRE(ctx && in && dy && dw_master, "sg_conv_wgrad_tc: NULL");
  int rc = tc_check(d, "sg_conv_wgrad_tc");
  if (rc != SG_OK) return rc;
  SG_REQUIRE(d->out_dt == d->in_dt, "sg_conv_wgrad_tc: dy must have the operand dtype (in_dt)");
  // fp32 operands are read as tf32: both operands are MN-major, which for 4-byte types exists only in the 32-byte-atom
  // flavour of the 128B swizzle (TMA SWIZZLE_128B_ATOM_32B + UMMA layout type SWIZZLE_128B_BASE32B)
  const CUtensorMapSwizzle swz = d->in_dt == SG_F32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  SG_REQUIRE(((uintptr_t)in & 15) == 0 && ((uintptr_t)dy & 15) == 0, "sg_conv_wgrad_tc: pointers must be 16-byte aligned");
  PFN_encodeTiled enc;
  rc = get_encode(ctx, &enc);
  if (rc != SG_OK) return rc;

  static_assert(sizeof(TcWgradParams) < 4000, "kernel parameter block too large");
  TcWgradParams p;
  memset(&p, 0, sizeof(p));
  const int es = d->in_dt == SG_F32 ? 4 : 2;
  const int KC = 128 / es, UK = 32 / es;
  p.ntaps = d->ntaps; p.c_in = d->c_in; p.c_out = d->c_out;
  p.w_ci_stride = d->w_ci_stride; p.w_co_stride = d->w_co_stride;
  p.dw = dw_master;
  p.db = db;
  p.db2 = db2;
  p.bias_partial = ctx->det_scratch + (SG_DET_SCRATCH_BYTES - (1u << 20)) / sizeof(float);      // last MB of the scratch
  p.sems = ctx->det_tickets;
  p.BN = d->c_in % 256 == 0 ? 256 : (d->c_in % 128 == 0 ? 128 : (d->c_in % 64 == 0 ? 64 : 32));
  p.ci_tiles = d->c_in / p.BN;
  p.co_tiles = sg_div_up(d->c_out, 128);
  p.a_chunks = 128 / KC;
  p.b_chunks = p.BN / KC;
  // pixels per k-block: keep a stage <= 48 KB so that >= 4 stages fit
  int max_rows = (48 * 1024) / (128 * (p.a_chunks + p.b_chunks));
  if (max_rows > 128) max_rows = 128;
  max_rows = max_rows / UK * UK;
  SG_REQUIRE(max_rows >= UK, "sg_conv_wgrad_tc: tile does not fit");
  choose_box(d->grid_w, d->grid_h, d->n, max_rows, UK, &p.TW, &p.TH, &p.TN);
  const int PR = p.TW * p.TH * p.TN;
  SG_REQUIRE(PR % UK == 0 && PR <= max_rows, "sg_conv_wgrad_tc: internal box choice error (%d)", PR);
  p.tiles_x = sg_div_up(d->grid_w, p.TW); p.tiles_y = sg_div_up(d->grid_h, p.TH); p.tiles_n = sg_div_up(d->n, p.TN);
  p.chunk_bytes = (uint32_t)PR * 128u;
  p.stage_stride = (uint32_t)(p.a_chunks + p.b_chunks) * p.chunk_bytes;
  p.stage_stride = (p.stage_stride + 1023u) & ~1023u;
  const uint32_t ones_bytes = db ? (uint32_t)PR * 128u : 0u;             // constant all-ones B tile of the bias units
  int stages = (int)((220u * 1024u - ones_bytes) / p.stage_stride);
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  SG_REQUIRE(stages >= 2, "sg_conv_wgrad_tc: not enough shared memory for 2 stages");
  p.stages = stages;

  const int ptiles = p.tiles_x * p.tiles_y * p.tiles_n;
  long long base_units = (long long)d->ntaps * p.co_tiles * p.ci_tiles;
  // pixel splits: static round-robin over #SMs persistent CTAs costs ceil(units / #SMs) unit-times, so pick the split
  // count whose last wave is fullest (e.g. 72 base units: 4 splits = 288 units = 1.95 waves, not 5 splits = 2.43 waves)
  int splits = wgrad_choose_splits(ptiles, base_units, p.co_tiles, ctx->num_sms);
  p.ptiles_per_split = sg_div_up(ptiles, splits);
  p.splits = sg_div_up(ptiles, p.ptiles_per_split);
  p.partial = ctx->det_scratch;
  // measured per layer (tools/bench_conv.py): ordered turns cost ~one epilogue per split on the critical path, which only long
  // main loops hide; the scratch + grid-barrier combine costs ~5-15 us flat
  p.det_mode = p.splits == 1 ? 0 : ((p.splits <= 4 && p.ptiles_per_split >= 64) ? 1 : 2);
  if (p.det_mode == 2 && (long long)base_units * p.splits * 128 * p.BN * (long long)sizeof(float) > (long long)SG_DET_SCRATCH_BYTES - (1 << 20)) {
    // the partial tiles would not fit the context's scratch: fall back to 4 ordered splits
    p.ptiles_per_split = sg_div_up(ptiles, 4);
    p.splits = sg_div_up(ptiles, p.ptiles_per_split);
    p.det_mode = p.splits == 1 ? 0 : 1;
  }

  bool used[4] = {false, false, false, false};
  for (int t = 0; t < d->ntaps; ++t) {
    int py = posmod(d->tap_dy[t], d->in_sy), px = posmod(d->tap_dx[t], d->in_sx);
    int v = py * 2 + px;
    p.tap_view[t] = v;
    p.tap_oy[t] = floordiv(d->tap_dy[t], d->in_sy);
    p.tap_ox[t] = floordiv(d->tap_dx[t], d->in_sx);
    p.tap_w_off[t] = d->tap_w_off[t];
    used[v] = true;
  }
  int first_used = -1;
  for (int v = 0; v < 4; ++v) {
    if (!used[v]) continue;
    if (first_used < 0) first_used = v;
    rc = encode_nhwc_view(enc, &p.map_in[v], d->in_dt, in, d->n, d->in_h, d->in_w, d->c_in, d->in_sy, d->in_sx, v / 2, v % 2, KC,
                          p.TW, p.TH, p.TN, swz);
    if (rc != SG_OK) return rc;
  }
  for (int v = 0; v < 4; ++v)
    if (!used[v]) p.map_in[v] = p.map_in[first_used];
  rc = encode_nhwc_view(enc, &p.map_dy, d->in_dt, dy, d->n, d->out_h, d->out_w, d->c_out, d->out_sy, d->out_sx, d->out_py,
                        d->out_px, KC, p.TW, p.TH, p.TN, swz);
  if (rc != SG_OK) return rc;

  long long units = base_units * p.splits + (db ? (long long)p.co_tiles * p.splits : 0);
  int grid = (int)(units < ctx->num_sms ? units : ctx->num_sms);
  size_t smem = (size_t)stages * p.stage_stride + 1024 + ones_bytes;
  // det_mode 2 ends in a grid-wide barrier: launched cooperatively, so the runtime guarantees (or refuses) co-residency
  if (d->in_dt == SG_F32) {
    SG_CHECK_CUDA(cudaFuncSetAttribute(k_wgrad_tc<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SG_CHECK_CUDA(sg_launch_ex(ctx, p.det_mode == 2, k_wgrad_tc<float>, grid, TC_THREADS, smem, p));
  } else {
    SG_CHECK_CUDA(cudaFuncSetAttribute(k_wgrad_tc<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SG_CHECK_CUDA(sg_launch_ex(ctx, p.det_mode == 2, k_wgrad_tc<__nv_bfloat16>, grid, TC_THREADS, smem, p));
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
