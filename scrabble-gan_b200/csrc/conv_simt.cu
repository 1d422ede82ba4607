// Exact-fp32 direct convolution family on the FFMA pipe (generic sg_conv_desc; see include/sgan.h).
// Used for (a) the edge layers that are not tensor-core shaped (K8: Cin=1 first convs, Cout=1 output conv,
// the C/8-channel attention projections) and (b) the "fp32" parity mode of the whole network.
// Reference ops replaced: Conv2D / Conv2DBackpropInput / Conv2DBackpropFilter / Conv2DTranspose
// (resnet_ops.py:57,65,69,98,103,109; net_architecture.py:28-49,283).
// Implicit GEMM with 64 x TN x 16 shared-memory tiles; K is the flattened (tap, ci) index so that Cin=1
// layers (K = 9) do not waste a 16-wide chunk per tap.
#include "common.cuh"

#define CS_TM 64
#define CS_TK 16

__device__ __forceinline__ float ld_any(const void* p, long long i, int dt) {
  return dt == SG_F32 ? reinterpret_cast<const float*>(p)[i] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
}
__device__ __forceinline__ void st_any(void* p, long long i, int dt, float v) {
  if (dt == SG_F32) reinterpret_cast<float*>(p)[i] = v;
  else reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------------------------------------------
// forward.  M = n*grid_h*grid_w output positions, N = c_out, K = ntaps*c_in.
// TN = 64: thread (tx,ty) computes 4 rows x 4 cols;  TN = 16: 4 rows x 1 col.
// ---------------------------------------------------------------------------------------------------
template <int TN, int RN>
__global__ void __launch_bounds__(256) k_conv_fwd_simt(sg_conv_desc d, const void* __restrict__ in,
                                                        const float* __restrict__ w, const float* __restrict__ bias,
                                                        const void* __restrict__ mask, void* __restrict__ out) {
  __shared__ float As[CS_TK][CS_TM + 4];
  __shared__ float Bs[CS_TK][TN + 4];
  constexpr int TX = TN / RN;                  // threads along N (16)
  const int tid = threadIdx.x;
  const int tx = tid % TX, ty = tid / TX;      // ty in [0,16)
  const long long M = (long long)d.n * d.grid_h * d.grid_w;
  const int K = d.ntaps * d.c_in;
  const long long m0 = (long long)blockIdx.x * CS_TM;
  const int n0 = blockIdx.y * TN;

  float acc[4][RN];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < RN; ++j) acc[i][j] = 0.f;

  // each thread loads 4 A elements per chunk: fixed (row, k-offset) assignment -> decode the pixel once
  // assignment: idx = tid + i*256, kk = idx % 16, mm = idx / 16  => mm = tid/16 + 16*i, kk = tid%16
  const int a_kk = tid % CS_TK;
  int a_n[4], a_y[4], a_x[4];
  bool a_ok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    long long gm = m0 + tid / CS_TK + 16 * i;
    a_ok[i] = gm < M;
    long long g = a_ok[i] ? gm : 0;
    a_x[i] = (int)(g % d.grid_w);
    g /= d.grid_w;
    a_y[i] = (int)(g % d.grid_h);
    a_n[i] = (int)(g / d.grid_h);
  }

  for (int k0 = 0; k0 < K; k0 += CS_TK) {
    {
      int gk = k0 + a_kk;
      bool kok = gk < K;
      int t = kok ? gk / d.c_in : 0, ci = kok ? gk % d.c_in : 0;
      int dy = d.tap_dy[t], dx = d.tap_dx[t];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float v = 0.f;
        if (kok && a_ok[i]) {
          int iy = a_y[i] * d.in_sy + dy, ix = a_x[i] * d.in_sx + dx;
          if (iy >= 0 && iy < d.in_h && ix >= 0 && ix < d.in_w)
            v = ld_any(in, (((long long)a_n[i] * d.in_h + iy) * d.in_w + ix) * d.c_in + ci, d.in_dt);
        }
        As[a_kk][tid / CS_TK + 16 * i] = v;
      }
    }
    for (int idx = tid; idx < CS_TK * TN; idx += 256) {
      int nn = idx % TN, kk = idx / TN;
      int gk = k0 + kk, gn = n0 + nn;
      float v = 0.f;
      if (gk < K && gn < d.c_out) {
        int t = gk / d.c_in, ci = gk % d.c_in;
        v = w[d.tap_w_off[t] + (long long)ci * d.w_ci_stride + (long long)gn * d.w_co_stride];
      }
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < CS_TK; ++kk) {
      float a[4], b[RN];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < RN; ++j) b[j] = Bs[kk][tx * RN + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < RN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    long long gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
    long long g = gm;
    int ox = (int)(g % d.grid_w);
    g /= d.grid_w;
    int oy = (int)(g % d.grid_h);
    int ni = (int)(g / d.grid_h);
    long long base = (((long long)ni * d.out_h + oy * d.out_sy + d.out_py) * d.out_w + ox * d.out_sx + d.out_px) * d.c_out;
#pragma unroll
    for (int j = 0; j < RN; ++j) {
      int gn = n0 + tx * RN + j;
      if (gn >= d.c_out) continue;
      float v = acc[i][j];
      if (bias) v += bias[gn];
      if (d.relu) v = fmaxf(v, 0.f);
      if (mask) v = ld_any(mask, base + gn, d.mask_dt) > 0.f ? v : 0.f;
      if (d.accumulate) v += ld_any(out, base + gn, d.out_dt);
      st_any(out, base + gn, d.out_dt, v);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// filter gradient.  M' = ntaps*c_in (flattened k index), N = c_out, reduction over output positions,
// split across gridDim.z; the splits of a tile add into dw in split order (ordered turns, common.cuh scheme A), so the
// result is bitwise repeatable (dw is accumulated into: caller zeroes it).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_conv_wgrad_simt(sg_conv_desc d, const void* __restrict__ in,
                                                          const void* __restrict__ dy, float* __restrict__ dw,
                                                          long long pos_per_split, unsigned int* __restrict__ sems) {
  __shared__ float As[CS_TK][CS_TM + 4];   // [pos][kflat]
  __shared__ float Bs[CS_TK][64 + 4];      // [pos][co]
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const long long P = (long long)d.n * d.grid_h * d.grid_w;
  const int KF = d.ntaps * d.c_in;
  const int kf0 = blockIdx.x * CS_TM;
  const int n0 = blockIdx.y * 64;
  const long long pbeg = (long long)blockIdx.z * pos_per_split;
  const long long pend = pbeg + pos_per_split < P ? pbeg + pos_per_split : P;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  // A loads: idx = tid + i*256 -> kf = idx % 64, pp = idx / 64 (4 positions per thread, fixed kf)
  const int a_kf = tid % CS_TM;
  const int gkf = kf0 + a_kf;
  const bool kf_ok = gkf < KF;
  const int a_t = kf_ok ? gkf / d.c_in : 0, a_ci = kf_ok ? gkf % d.c_in : 0;
  const int a_dy = d.tap_dy[a_t], a_dx = d.tap_dx[a_t];

  for (long long p0 = pbeg; p0 < pend; p0 += CS_TK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int pp = tid / CS_TM + 4 * i;
      long long gp = p0 + pp;
      float v = 0.f;
      if (kf_ok && gp < pend) {
        long long g = gp;
        int ox = (int)(g % d.grid_w);
        g /= d.grid_w;
        int oy = (int)(g % d.grid_h);
        int ni = (int)(g / d.grid_h);
        int iy = oy * d.in_sy + a_dy, ix = ox * d.in_sx + a_dx;
        if (iy >= 0 && iy < d.in_h && ix >= 0 && ix < d.in_w)
          v = ld_any(in, (((long long)ni * d.in_h + iy) * d.in_w + ix) * d.c_in + a_ci, d.in_dt);
      }
      As[pp][a_kf] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int idx = tid + i * 256;
      int nn = idx % 64, pp = idx / 64;
      long long gp = p0 + pp;
      int gn = n0 + nn;
      float v = 0.f;
      if (gp < pend && gn < d.c_out) {
        long long g = gp;
        int ox = (int)(g % d.grid_w);
        g /= d.grid_w;
        int oy = (int)(g % d.grid_h);
        int ni = (int)(g / d.grid_h);
        v = ld_any(dy, (((long long)ni * d.out_h + oy * d.out_sy + d.out_py) * d.out_w + ox * d.out_sx + d.out_px) * d.c_out + gn,
                   d.out_dt);
      }
      Bs[pp][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < CS_TK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  unsigned int* sem = sems + (long long)blockIdx.y * gridDim.x + blockIdx.x;
  if (gridDim.z > 1) {
    if (tid == 0) sg_turn_wait(sem, blockIdx.z);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int kf = kf0 + ty * 4 + i;
    if (kf >= KF) continue;
    int t = kf / d.c_in, ci = kf % d.c_in;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int gn = n0 + tx * 4 + j;
      if (gn >= d.c_out) continue;
      atomicAdd(dw + d.tap_w_off[t] + (long long)ci * d.w_ci_stride + (long long)gn * d.w_co_stride, acc[i][j]);
    }
  }
  if (gridDim.z > 1) {
    __syncthreads();
    if (tid == 0) sg_turn_pass(sem, blockIdx.z, gridDim.z);
  }
}

// ---------------------------------------------------------------------------------------------------
// Edge-layer specialisations (K8).  The image-side layers (Cin = 1: D/W/style B1.conv1 + shortcut, R.conv1) and the
// single-channel output conv (Cout = 1: G.out, and the input gradients of the Cin = 1 layers) have a huge pixel
// count but K = 9 or N = 1: they are HBM-bound streaming kernels, not GEMMs.
// ---------------------------------------------------------------------------------------------------
struct Pix { int n, y, x; };
__device__ __forceinline__ Pix decode_pix(long long p, int gh, int gw) {
  Pix r;
  r.x = (int)(p % gw);
  p /= gw;
  r.y = (int)(p % gh);
  r.n = (int)(p / gh);
  return r;
}

// filter gradient with ONE narrow side: WIDE = number of channels on the wide side (<= 256, divides 256).
//   NARROW_IN  (c_in == 1): dW[t][co] += sum_p in[p + tap_t] * dy[p, co]      thread <-> co
//   !NARROW_IN (c_out == 1): dW[t][ci] += sum_p in[p + tap_t, ci] * dy[p]     thread <-> ci
template <bool NARROW_IN>
__global__ void __launch_bounds__(256) k_wgrad_narrow(sg_conv_desc d, const void* __restrict__ in, const void* __restrict__ dy,
                                                       float* __restrict__ dw, long long pos_per_block, float* __restrict__ scratch,
                                                       unsigned int* __restrict__ ticket) {
  extern __shared__ float red[];                       // [lanes][ntaps][wide]
  const int wide = NARROW_IN ? d.c_out : d.c_in;
  const int lanes = 256 / wide;
  const int ch = threadIdx.x % wide, lane = threadIdx.x / wide;
  const long long P = (long long)d.n * d.grid_h * d.grid_w;
  const long long p0 = (long long)blockIdx.x * pos_per_block;
  const long long p1 = p0 + pos_per_block < P ? p0 + pos_per_block : P;
  float acc[SG_MAX_TAPS];
#pragma unroll
  for (int t = 0; t < SG_MAX_TAPS; ++t) acc[t] = 0.f;
  if (lane < lanes) {
    for (long long p = p0 + lane; p < p1; p += lanes) {
      Pix q = decode_pix(p, d.grid_h, d.grid_w);
      long long opix = ((long long)q.n * d.out_h + q.y) * d.out_w + q.x;
      float dyv = NARROW_IN ? ld_any(dy, opix * d.c_out + ch, d.out_dt) : ld_any(dy, opix, d.out_dt);
#pragma unroll
      for (int t = 0; t < SG_MAX_TAPS; ++t) {
        if (t < d.ntaps) {
          int iy = q.y + d.tap_dy[t], ix = q.x + d.tap_dx[t];
          if (iy >= 0 && iy < d.in_h && ix >= 0 && ix < d.in_w) {
            long long ipix = ((long long)q.n * d.in_h + iy) * d.in_w + ix;
            float xv = NARROW_IN ? ld_any(in, ipix, d.in_dt) : ld_any(in, ipix * d.c_in + ch, d.in_dt);
            acc[t] = fmaf(xv, dyv, acc[t]);
          }
        }
      }
    }
#pragma unroll
    for (int t = 0; t < SG_MAX_TAPS; ++t)
      if (t < d.ntaps) red[((long long)lane * d.ntaps + t) * wide + ch] = acc[t];
  }
  __syncthreads();
  // deterministic combine (common.cuh, scheme B): per-block partial filters, summed in block order by the last block
  const int nout = d.ntaps * wide;
  for (int i = threadIdx.x; i < nout; i += 256) {
    int t = i / wide, c = i % wide;
    float sum = 0.f;
    for (int l = 0; l < lanes; ++l) sum += red[((long long)l * d.ntaps + t) * wide + c];
    scratch[(long long)blockIdx.x * nout + i] = sum;
  }
  sg_det_finish(scratch, scratch + (long long)gridDim.x * nout, ticket, gridDim.x, blockIdx.x, nout, [&](int i, float sum) {
    int t = i / wide, c = i % wide;
    long long off = d.tap_w_off[t] + (NARROW_IN ? (long long)c * d.w_co_stride : (long long)c * d.w_ci_stride);
    dw[off] += sum;
  });
}

__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  float4 a = sg_ld4(p), b = sg_ld4(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) {
  float4 a = sg_ld4(p), b = sg_ld4(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// forward-type conv with c_out == 1 and c_in % 8 == 0 (c_in/8 a power of two <= 32): c_in/8 threads per output
// pixel, each holding its 8 channels x ntaps weights in registers; shuffle reduction; full epilogue.
template <typename TIn>
__global__ void __launch_bounds__(256, 4) k_conv_fwd_cout1(sg_conv_desc d, const TIn* __restrict__ in, const float* __restrict__ w,
                                                            const float* __restrict__ bias, const void* __restrict__ mask,
                                                            void* __restrict__ out) {
  // the ntaps x c_in filter lives in shared memory (2 broadcast LDS.128 per tap) instead of 72 registers per thread:
  // 4 blocks per SM instead of 2, which is what hides the load latency of this streaming kernel
  __shared__ __align__(16) float ws[9][256];
  const int tpp = d.c_in / 8;                            // threads per pixel
  const int sub = threadIdx.x % tpp;
  const int pix_per_block = 256 / tpp;
  for (int i = threadIdx.x; i < 9 * d.c_in; i += 256) {
    int t = i / d.c_in, ci = i - t * d.c_in;
    ws[t][ci] = (t < d.ntaps) ? w[d.tap_w_off[t] + (long long)ci * d.w_ci_stride] : 0.f;
  }
  __syncthreads();
  const float b0 = bias ? bias[0] : 0.f;
  // one output row per block iteration (no per-pixel integer division); all lanes of a warp stay in the loop together
  // because the shuffle reduction needs the full c_in/8 group
  const int nrows = d.n * d.grid_h;
  const int px_lane = threadIdx.x / tpp;
  const int xsteps = (d.grid_w + pix_per_block - 1) / pix_per_block;
  for (int row = blockIdx.x; row < nrows; row += gridDim.x) {
    const int ni = row / d.grid_h, y = row - ni * d.grid_h;
    const TIn* img = in + (long long)ni * d.in_h * d.in_w * d.c_in + sub * 8;
    for (int xs = 0; xs < xsteps; ++xs) {
      const int x = px_lane + xs * pix_per_block;
      const bool live = x < d.grid_w;
      float acc = 0.f;
      if (live) {
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          if (t < d.ntaps) {
            int iy = y * d.in_sy + d.tap_dy[t], ix = x * d.in_sx + d.tap_dx[t];
            if (iy >= 0 && iy < d.in_h && ix >= 0 && ix < d.in_w) {
              float v[8];
              load8(img + (iy * d.in_w + ix) * d.c_in, v);
              const float4 w0 = *reinterpret_cast<const float4*>(&ws[t][sub * 8]), w1 = *reinterpret_cast<const float4*>(&ws[t][sub * 8 + 4]);
              acc = fmaf(v[0], w0.x, acc); acc = fmaf(v[1], w0.y, acc); acc = fmaf(v[2], w0.z, acc); acc = fmaf(v[3], w0.w, acc);
              acc = fmaf(v[4], w1.x, acc); acc = fmaf(v[5], w1.y, acc); acc = fmaf(v[6], w1.z, acc); acc = fmaf(v[7], w1.w, acc);
            }
          }
        }
      }
      for (int o = tpp >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (live && sub == 0) {
        long long idx = ((long long)ni * d.out_h + y * d.out_sy + d.out_py) * d.out_w + x * d.out_sx + d.out_px;
        float v = acc + b0;
        if (d.relu) v = fmaxf(v, 0.f);
        if (mask) v = ld_any(mask, idx, d.mask_dt) > 0.f ? v : 0.f;
        if (d.accumulate) v += ld_any(out, idx, d.out_dt);
        st_any(out, idx, d.out_dt, v);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Edge layers, second generation: C = 64 on the wide side, shared-memory staged.
// ---------------------------------------------------------------------------------------------------
// Filter gradient with one single-channel side as a skinny GEMM over pixels:
//     dW[t][c] += sum_p wide[p, c] * narrow[p + off_t]            (c < 64, t < ntaps <= 9)
//   c_in == 1 : wide = dy [n,H,W,64], narrow = layer input,  off_t = +tap_t
//   c_out == 1: wide = layer input [n,H,W,64], narrow = dy,   off_t = -tap_t
// Block = 192 threads = 64 channels x 3 tap groups; a chunk of 64 pixels of the wide tensor is staged in shared memory
// (coalesced 16-byte loads) together with the 9 x 64 patch of the narrow tensor; each thread then runs 4 pixels per
// step (4 scalar LDS of its channel + 3 broadcast LDS.128 of the patch -> 12 FMA).
#define WN_PIX 64
template <typename TW>
__global__ void __launch_bounds__(192) k_wgrad_narrow64(const TW* __restrict__ wide, const void* __restrict__ narrow, int narrow_dt,
                                                         int n, int H, int W, int nH, int nW, int ntaps, sg_conv_desc d,
                                                         int sign, float* __restrict__ dw, long long chunks_per_block,
                                                         int narrow_in, float* __restrict__ scratch, unsigned int* __restrict__ ticket) {
  __shared__ float Bs[WN_PIX][64];
  __shared__ __align__(16) float As[9][WN_PIX];
  const int tid = threadIdx.x;
  const int c = tid & 63, tg = tid >> 6;
  const long long P = (long long)n * H * W;
  const long long nchunks = (P + WN_PIX - 1) / WN_PIX;
  long long ch0 = (long long)blockIdx.x * chunks_per_block, ch1 = ch0 + chunks_per_block;
  if (ch1 > nchunks) ch1 = nchunks;
  float acc[3] = {0.f, 0.f, 0.f};
  for (long long chk = ch0; chk < ch1; ++chk) {
    const long long p0 = chk * WN_PIX;
    const int cnt = P - p0 < WN_PIX ? (int)(P - p0) : WN_PIX;
    __syncthreads();
    // wide tile: cnt x 64 contiguous elements
    {
      const TW* src = wide + p0 * 64;
      for (int i = tid; i < WN_PIX * 64 / 4; i += 192) {
        int e = i * 4, px = e >> 6, cc = e & 63;
        float4 v = px < cnt ? sg_ld4(src + e) : make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(&Bs[px][cc]) = v;
      }
    }
    // narrow patch: 9 x 64 values
    for (int i = tid; i < 9 * WN_PIX; i += 192) {
      int t = i / WN_PIX, px = i % WN_PIX;
      float v = 0.f;
      if (t < ntaps && px < cnt) {
        Pix q = decode_pix(p0 + px, H, W);
        int y = q.y + sign * d.tap_dy[t], x = q.x + sign * d.tap_dx[t];
        if (y >= 0 && y < nH && x >= 0 && x < nW) v = ld_any(narrow, ((long long)q.n * nH + y) * nW + x, narrow_dt);
      }
      As[t][px] = v;
    }
    __syncthreads();
    if (3 * tg < ntaps) {
#pragma unroll 4
      for (int px = 0; px < WN_PIX; px += 4) {
        float b0 = Bs[px][c], b1 = Bs[px + 1][c], b2 = Bs[px + 2][c], b3 = Bs[px + 3][c];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          float4 a = *reinterpret_cast<const float4*>(&As[3 * tg + j][px]);
          acc[j] = fmaf(a.x, b0, acc[j]); acc[j] = fmaf(a.y, b1, acc[j]);
          acc[j] = fmaf(a.z, b2, acc[j]); acc[j] = fmaf(a.w, b3, acc[j]);
        }
      }
    }
  }
  // deterministic combine (common.cuh, scheme B): slot = [9 taps][64 channels] per block
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    int t = 3 * tg + j;
    if (t < 9) scratch[(long long)blockIdx.x * 576 + t * 64 + c] = (t < ntaps) ? acc[j] : 0.f;
  }
  sg_det_finish(scratch, scratch + (long long)gridDim.x * 576, ticket, gridDim.x, blockIdx.x, 576, [&](int i, float sum) {
    int t = i >> 6, cc = i & 63;
    if (t >= ntaps) return;
    long long off = d.tap_w_off[t] + (narrow_in ? (long long)cc * d.w_co_stride : (long long)cc * d.w_ci_stride);
    dw[off] += sum;
  });
}

// forward conv with c_in == 1, c_out % 8 == 0 (<= 64 per pixel group), unit strides: 8 output channels per thread with
// their ntaps x 8 weights in registers; the input patch comes through L1 (neighbouring threads share it); 16/32-byte
// vector stores.  out = act(bias + sum_t x[p + tap_t] * w[t, :]) (+ out when accumulate).
template <typename TOut, int CH>
__global__ void __launch_bounds__(256, 4) k_conv_fwd_cin1(sg_conv_desc d, const float* __restrict__ in, const float* __restrict__ w,
                                                           const float* __restrict__ bias, TOut* __restrict__ out) {
  // CH output channels per thread: the 3x3 input patch is loaded ONCE per (pixel, CH channels) and reused for CH/8 chunks
  // of 8 channels (this kernel is instruction bound: with CH = 8 the nine patch loads and their bounds checks were
  // repeated for every 8 channels)
  __shared__ __align__(16) float ws[10][256];          // 9 taps + bias row, c_out <= 256
  const int groups = d.c_out / CH;                     // threads per pixel
  const int sub = threadIdx.x % groups;
  const int pix_per_block = 256 / groups;
  for (int i = threadIdx.x; i < 10 * d.c_out; i += 256) {
    int t = i / d.c_out, co = i - t * d.c_out;
    float v = 0.f;
    if (t < d.ntaps) v = w[d.tap_w_off[t] + (long long)co * d.w_co_stride];
    else if (t == 9 && bias) v = bias[co];
    ws[t][co] = v;
  }
  __syncthreads();
  // pixels are linearised over (image, y, x) with 32-bit index math (two divisions per ~400 instructions of work)
  const int total = d.n * d.grid_h * d.grid_w;
  const int px_lane = threadIdx.x / groups;
  for (int p = blockIdx.x * pix_per_block + px_lane; p < total; p += gridDim.x * pix_per_block) {
    const int x = p % d.grid_w, row = p / d.grid_w;
    const int ni = row / d.grid_h, y = row - ni * d.grid_h;
    const float* img = in + (long long)ni * d.in_h * d.in_w;
    TOut* orow = out + ((long long)ni * d.out_h + y) * d.out_w * d.c_out;
    {
      float xv[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        xv[t] = 0.f;
        if (t < d.ntaps) {
          int iy = y + d.tap_dy[t], ix = x + d.tap_dx[t];
          if (iy >= 0 && iy < d.in_h && ix >= 0 && ix < d.in_w) xv[t] = __ldg(img + iy * d.in_w + ix);
        }
      }
      TOut* op = orow + x * d.c_out + sub * CH;
#pragma unroll
      for (int c8 = 0; c8 < CH; c8 += 8) {
        const int cb = sub * CH + c8;
        float acc[8];
        {
          const float4 b0 = *reinterpret_cast<const float4*>(&ws[9][cb]), b1 = *reinterpret_cast<const float4*>(&ws[9][cb + 4]);
          acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w; acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          if (t < d.ntaps) {
            const float4 w0 = *reinterpret_cast<const float4*>(&ws[t][cb]), w1 = *reinterpret_cast<const float4*>(&ws[t][cb + 4]);
            acc[0] = fmaf(xv[t], w0.x, acc[0]); acc[1] = fmaf(xv[t], w0.y, acc[1]); acc[2] = fmaf(xv[t], w0.z, acc[2]); acc[3] = fmaf(xv[t], w0.w, acc[3]);
            acc[4] = fmaf(xv[t], w1.x, acc[4]); acc[5] = fmaf(xv[t], w1.y, acc[5]); acc[6] = fmaf(xv[t], w1.z, acc[6]); acc[7] = fmaf(xv[t], w1.w, acc[7]);
          }
        }
        if (d.relu) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = fmaxf(acc[j], 0.f);
        }
        if (d.accumulate) {
          float4 a = sg_ld4(op + c8), b = sg_ld4(op + c8 + 4);
          acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w; acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
        }
        sg_st4(op + c8, make_float4(acc[0], acc[1], acc[2], acc[3]));
        sg_st4(op + c8 + 4, make_float4(acc[4], acc[5], acc[6], acc[7]));
      }
    }
  }
}


// ---------------------------------------------------------------------------------------------------
// Edge layers, third generation (C = 64 on the wide side, 3x3 "same" or 1x1, unit strides): 4 consecutive pixels x 8
// channels per thread.  ncu on the second-generation kernels (profiles/r02_edge_kernels_ncu.md) showed the L1/LSU path at
// 60-80 % -- k_conv_fwd_cout1 re-read each input pixel once per tap with two 8-byte loads, k_conv_fwd_cin1<.,32> wrote its
// 64 bf16 channels with 8-byte stores at a 64-byte lane stride (16 wavefronts per store) -- while DRAM sat at 5-10 %.  Here
// a thread keeps a 3 x 6 pixel patch in registers for its 4 outputs (each input pixel is loaded 1.5 times, not 9), every
// global access is a 16-byte vector per lane, and the 8 threads of a pixel quad cover the 64 channels of a pixel
// contiguously (full 128-byte lines).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ld8f(const float* p, float (&v)[8]) {
  float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld8f(const __nv_bfloat16* p, float (&v)[8]) {
  uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float2 f = __bfloat1622float2(h[j]);
    v[2 * j] = f.x; v[2 * j + 1] = f.y;
  }
}
__device__ __forceinline__ void st8f(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *(reinterpret_cast<float4*>(p) + 1) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void st8f(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 r;
  __nv_bfloat162 h;
  h = __floats2bfloat162_rn(v[0], v[1]); r.x = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[2], v[3]); r.y = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[4], v[5]); r.z = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(v[6], v[7]); r.w = *reinterpret_cast<uint32_t*>(&h);
  *reinterpret_cast<uint4*>(p) = r;
}

// taps of a 3x3 "same" / 1x1 conv as a dense 3 x 3 table: slot (dy + 1) * 3 + (dx + 1) -> tap index or -1
struct EdgeTaps { int slot[9]; };

// c_out == 1, c_in == 64: out[p] = act(b + sum_{t, c} in[p + tap_t, c] * w[t, c])
template <typename TIn>
__global__ void __launch_bounds__(256, 3) k_conv_fwd_cout1_q4(sg_conv_desc d, EdgeTaps tp, const TIn* __restrict__ in, const float* __restrict__ w,
                                                               const float* __restrict__ bias, const void* __restrict__ mask,
                                                               void* __restrict__ out) {
  __shared__ __align__(16) float ws[9][64];               // dense 3 x 3 slots (zero where the conv has no tap)
  for (int i = threadIdx.x; i < 9 * 64; i += 256) {
    int sl = i / 64, ci = i - sl * 64;
    int t = tp.slot[sl];
    ws[sl][ci] = t >= 0 ? w[d.tap_w_off[t] + (long long)ci * d.w_ci_stride] : 0.f;
  }
  __syncthreads();
  const float b0 = bias ? bias[0] : 0.f;
  const int oct = threadIdx.x & 7;                         // channel octet of this thread
  const int quads_x = d.grid_w >> 2;
  const long long nquads = (long long)d.n * d.grid_h * quads_x;
  for (long long q = (long long)blockIdx.x * 32 + (threadIdx.x >> 3); q < nquads; q += (long long)gridDim.x * 32) {
    const int xq = (int)(q % quads_x);
    const long long row = q / quads_x;
    const int y = (int)(row % d.grid_h);
    const long long ni = row / d.grid_h;
    const int x0 = xq * 4;
    const TIn* img = in + ni * d.in_h * d.in_w * 64 + oct * 8;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int iy = y + r - 1;
      if (iy < 0 || iy >= d.in_h) continue;
      if (r != 1 && tp.slot[3 * r] < 0 && tp.slot[3 * r + 1] < 0 && tp.slot[3 * r + 2] < 0) continue;
      float v[6][8];
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        const int ix = x0 + j - 1;
        if (ix >= 0 && ix < d.in_w) ld8f(img + ((long long)iy * d.in_w + ix) * 64, v[j]);
        else {
#pragma unroll
          for (int c = 0; c < 8; ++c) v[j][c] = 0.f;
        }
      }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const float4 w0 = *reinterpret_cast<const float4*>(&ws[3 * r + dx][oct * 8]), w1 = *reinterpret_cast<const float4*>(&ws[3 * r + dx][oct * 8 + 4]);
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const float (&u)[8] = v[px + dx];
          float a = acc[px];
          a = fmaf(u[0], w0.x, a); a = fmaf(u[1], w0.y, a); a = fmaf(u[2], w0.z, a); a = fmaf(u[3], w0.w, a);
          a = fmaf(u[4], w1.x, a); a = fmaf(u[5], w1.y, a); a = fmaf(u[6], w1.z, a); a = fmaf(u[7], w1.w, a);
          acc[px] = a;
        }
      }
    }
#pragma unroll
    for (int px = 0; px < 4; ++px) {
      acc[px] += __shfl_xor_sync(0xffffffffu, acc[px], 1);
      acc[px] += __shfl_xor_sync(0xffffffffu, acc[px], 2);
      acc[px] += __shfl_xor_sync(0xffffffffu, acc[px], 4);
    }
    if (oct < 4) {                                         // thread `oct` of the quad finishes pixel x0 + oct
      float vv = (oct == 0 ? acc[0] : oct == 1 ? acc[1] : oct == 2 ? acc[2] : acc[3]) + b0;
      const long long idx = (ni * d.out_h + y) * d.out_w + x0 + oct;
      if (d.relu) vv = fmaxf(vv, 0.f);
      if (mask) vv = ld_any(mask, idx, d.mask_dt) > 0.f ? vv : 0.f;
      if (d.accumulate) vv += ld_any(out, idx, d.out_dt);
      st_any(out, idx, d.out_dt, vv);
    }
  }
}

// c_in == 1 (fp32 input), c_out == 64: out[p, :] = act(b + sum_t in[p + tap_t] * w[t, :]) (+ out when accumulate)
template <typename TOut>
__global__ void __launch_bounds__(256, 3) k_conv_fwd_cin1_q4(sg_conv_desc d, EdgeTaps tp, const float* __restrict__ in, const float* __restrict__ w,
                                                              const float* __restrict__ bias, TOut* __restrict__ out) {
  __shared__ __align__(16) float ws[10][64];              // dense 3 x 3 slots + bias row
  for (int i = threadIdx.x; i < 10 * 64; i += 256) {
    int sl = i / 64, co = i - sl * 64;
    float v = 0.f;
    if (sl < 9) {
      int t = tp.slot[sl];
      if (t >= 0) v = w[d.tap_w_off[t] + (long long)co * d.w_co_stride];
    } else if (bias) v = bias[co];
    ws[sl][co] = v;
  }
  __syncthreads();
  const int oct = threadIdx.x & 7;
  const int quads_x = d.grid_w >> 2;
  const long long nquads = (long long)d.n * d.grid_h * quads_x;
  for (long long q = (long long)blockIdx.x * 32 + (threadIdx.x >> 3); q < nquads; q += (long long)gridDim.x * 32) {
    const int xq = (int)(q % quads_x);
    const long long row = q / quads_x;
    const int y = (int)(row % d.grid_h);
    const long long ni = row / d.grid_h;
    const int x0 = xq * 4;
    const float* img = in + ni * d.in_h * d.in_w;
    float acc[4][8];
    {
      const float4 b0 = *reinterpret_cast<const float4*>(&ws[9][oct * 8]), b1 = *reinterpret_cast<const float4*>(&ws[9][oct * 8 + 4]);
#pragma unroll
      for (int px = 0; px < 4; ++px) {
        acc[px][0] = b0.x; acc[px][1] = b0.y; acc[px][2] = b0.z; acc[px][3] = b0.w;
        acc[px][4] = b1.x; acc[px][5] = b1.y; acc[px][6] = b1.z; acc[px][7] = b1.w;
      }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int iy = y + r - 1;
      if (iy < 0 || iy >= d.in_h) continue;
      if (r != 1 && tp.slot[3 * r] < 0 && tp.slot[3 * r + 1] < 0 && tp.slot[3 * r + 2] < 0) continue;
      float xv[6];
      {
        // x0 is a multiple of 4 and the row starts 16-byte aligned: one float4 for the 4 centre pixels + the two neighbours
        const float* rp = img + (long long)iy * d.in_w + x0;
        float4 c4 = __ldg(reinterpret_cast<const float4*>(rp));
        xv[1] = c4.x; xv[2] = c4.y; xv[3] = c4.z; xv[4] = c4.w;
        xv[0] = x0 > 0 ? __ldg(rp - 1) : 0.f;
        xv[5] = x0 + 4 < d.in_w ? __ldg(rp + 4) : 0.f;
      }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const float4 w0 = *reinterpret_cast<const float4*>(&ws[3 * r + dx][oct * 8]), w1 = *reinterpret_cast<const float4*>(&ws[3 * r + dx][oct * 8 + 4]);
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const float xs = xv[px + dx];
          acc[px][0] = fmaf(xs, w0.x, acc[px][0]); acc[px][1] = fmaf(xs, w0.y, acc[px][1]); acc[px][2] = fmaf(xs, w0.z, acc[px][2]);
          acc[px][3] = fmaf(xs, w0.w, acc[px][3]); acc[px][4] = fmaf(xs, w1.x, acc[px][4]); acc[px][5] = fmaf(xs, w1.y, acc[px][5]);
          acc[px][6] = fmaf(xs, w1.z, acc[px][6]); acc[px][7] = fmaf(xs, w1.w, acc[px][7]);
        }
      }
    }
    TOut* op = out + ((ni * d.out_h + y) * d.out_w + x0) * 64 + oct * 8;
#pragma unroll
    for (int px = 0; px < 4; ++px) {
      if (d.relu) {
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[px][c] = fmaxf(acc[px][c], 0.f);
      }
      if (d.accumulate) {
        float pv[8];
        ld8f(op + px * 64, pv);
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[px][c] += pv[c];
      }
      st8f(op + px * 64, acc[px]);
    }
  }
}

// Filter gradient of the same edge layers (see k_wgrad_narrow64 for the algebra): dW[t][c] += sum_p wide[p, c] * narrow[p + s * tap_t].
// 4 pixels x 8 channels per thread with all 9 x 8 partial filter entries in registers: per quad 4 vector loads of the wide
// tensor, a 3 x 6 patch of the narrow one and 288 FMA, no shared-memory staging and no barriers inside the pixel loop; the
// block then folds its 32 quad lanes (shuffles, one shared-memory pass) into ONE [9][64] partial for the ordered combine.
// tp.slot holds the tap of the patch position (s * dy + 1) * 3 + (s * dx + 1).
template <typename TW>
__global__ void __launch_bounds__(256, 2) k_wgrad_edge_q4(const TW* __restrict__ wide, const void* __restrict__ narrow, int narrow_dt, int n, int H,
                                                           int W, EdgeTaps tp, sg_conv_desc d, float* __restrict__ dw, int narrow_in,
                                                           float* __restrict__ scratch, unsigned int* __restrict__ ticket) {
  __shared__ float red[8][576];
  const int oct = threadIdx.x & 7;
  const int quads_x = W >> 2;
  const long long nquads = (long long)n * H * quads_x;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[t][c] = 0.f;
  bool row_used[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) row_used[r] = tp.slot[3 * r] >= 0 || tp.slot[3 * r + 1] >= 0 || tp.slot[3 * r + 2] >= 0;
  for (long long q = (long long)blockIdx.x * 32 + (threadIdx.x >> 3); q < nquads; q += (long long)gridDim.x * 32) {
    const int xq = (int)(q % quads_x);
    const long long row = q / quads_x;
    const int y = (int)(row % H);
    const long long ni = row / H;
    const int x0 = xq * 4;
    float wv[4][8];
    {
      const TW* wp = wide + ((ni * H + y) * W + x0) * 64 + oct * 8;
#pragma unroll
      for (int px = 0; px < 4; ++px) ld8f(wp + px * 64, wv[px]);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int iy = y + r - 1;
      if (!row_used[r] || iy < 0 || iy >= H) continue;
      float xv[6];
      const long long rb = (ni * H + iy) * W + x0;
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        const int ix = x0 + j - 1;
        xv[j] = (ix >= 0 && ix < W) ? ld_any(narrow, rb + j - 1, narrow_dt) : 0.f;
      }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const float xs = xv[px + dx];
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[3 * r + dx][c] = fmaf(xs, wv[px][c], acc[3 * r + dx][c]);
        }
      }
    }
  }
  // fold the 4 quads of the warp (lanes with equal oct), then the 8 warps through shared memory
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float v = acc[t][c];
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if (lane < 8) red[warp][t * 64 + oct * 8 + c] = v;
    }
  __syncthreads();
  for (int i = threadIdx.x; i < 576; i += 256) {
    float sum = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) sum += red[w8][i];
    scratch[(long long)blockIdx.x * 576 + i] = sum;
  }
  sg_det_finish(scratch, scratch + (long long)gridDim.x * 576, ticket, gridDim.x, blockIdx.x, 576, [&](int i, float sum) {
    const int sl = i >> 6, cc = i & 63;
    const int t = tp.slot[sl];
    if (t < 0) return;
    long long off = d.tap_w_off[t] + (narrow_in ? (long long)cc * d.w_co_stride : (long long)cc * d.w_ci_stride);
    dw[off] += sum;
  });
}

// true (and the slot table filled) when the conv is a unit-stride 3x3-"same"-like or 1x1 stencil on equal input / output grids
static bool edge_taps(const sg_conv_desc* d, EdgeTaps* tp) {
  if (!(d->in_sy == 1 && d->in_sx == 1 && d->out_sy == 1 && d->out_sx == 1 && d->out_py == 0 && d->out_px == 0)) return false;
  if (d->in_h != d->grid_h || d->in_w != d->grid_w || d->out_h != d->grid_h || d->out_w != d->grid_w || d->grid_w % 4 != 0) return false;
  for (int i = 0; i < 9; ++i) tp->slot[i] = -1;
  for (int t = 0; t < d->ntaps; ++t) {
    int dy = d->tap_dy[t], dx = d->tap_dx[t];
    if (dy < -1 || dy > 1 || dx < -1 || dx > 1) return false;
    int sl = (dy + 1) * 3 + dx + 1;
    if (tp->slot[sl] >= 0) return false;
    tp->slot[sl] = t;
  }
  return true;
}

static int check_desc(const sg_conv_desc* d, const char* who) {
  SG_REQUIRE(d != nullptr, "%s: desc is NULL", who);
  SG_REQUIRE(d->n >= 0 && d->in_h > 0 && d->in_w > 0 && d->c_in > 0 && d->out_h > 0 && d->out_w > 0 && d->c_out > 0,
             "%s: bad tensor dims", who);
  SG_REQUIRE(d->grid_h > 0 && d->grid_w > 0 && d->ntaps >= 1 && d->ntaps <= SG_MAX_TAPS, "%s: bad grid/taps", who);
  SG_REQUIRE(d->in_sy >= 1 && d->in_sx >= 1 && d->out_sy >= 1 && d->out_sx >= 1, "%s: bad strides", who);
  SG_REQUIRE((d->grid_h - 1) * d->out_sy + d->out_py < d->out_h && (d->grid_w - 1) * d->out_sx + d->out_px < d->out_w &&
                 d->out_py >= 0 && d->out_px >= 0,
             "%s: output placement exceeds the output tensor", who);
  SG_REQUIRE((d->in_dt == SG_F32 || d->in_dt == SG_BF16) && (d->out_dt == SG_F32 || d->out_dt == SG_BF16), "%s: bad dtype", who);
  return SG_OK;
}

extern "C" {

int sg_conv_fwd_simt(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const float* w_master, const float* bias,
                     const void* mask, void* out) {
  SG_REQUIRE(ctx && in && w_master && out, "sg_conv_fwd_simt: NULL");
  int rc = check_desc(d, "sg_conv_fwd_simt");
  if (rc != SG_OK) return rc;
  long long M = (long long)d->n * d->grid_h * d->grid_w;
  if (M == 0) return SG_OK;
  {
    EdgeTaps tp;
    const bool q4 = M < (1LL << 40) && edge_taps(d, &tp);
    if (q4 && d->c_out == 1 && d->c_in == 64 && ((uintptr_t)in & 15) == 0) {
      long long need = (M / 4 + 31) / 32, cap = (long long)ctx->num_sms * 12;
      int grid = (int)(need < cap ? need : cap);
      if (d->in_dt == SG_F32) sg_launch(ctx, k_conv_fwd_cout1_q4<float>, grid, 256, 0, *d, tp, (const float*)in, w_master, bias, mask, out);
      else sg_launch(ctx, k_conv_fwd_cout1_q4<__nv_bfloat16>, grid, 256, 0, *d, tp, (const __nv_bfloat16*)in, w_master, bias, mask, out);
      SG_POST_LAUNCH(ctx);
      return SG_OK;
    }
    if (q4 && d->c_in == 1 && d->c_out == 64 && d->in_dt == SG_F32 && !mask && ((uintptr_t)out & 15) == 0 && ((uintptr_t)in & 15) == 0) {
      long long need = (M / 4 + 31) / 32, cap = (long long)ctx->num_sms * 12;
      int grid = (int)(need < cap ? need : cap);
      if (d->out_dt == SG_F32) sg_launch(ctx, k_conv_fwd_cin1_q4<float>, grid, 256, 0, *d, tp, (const float*)in, w_master, bias, (float*)out);
      else sg_launch(ctx, k_conv_fwd_cin1_q4<__nv_bfloat16>, grid, 256, 0, *d, tp, (const float*)in, w_master, bias, (__nv_bfloat16*)out);
      SG_POST_LAUNCH(ctx);
      return SG_OK;
    }
  }
  {
    int tpp = d->c_in / 8;
    bool pow2 = tpp >= 1 && tpp <= 32 && (tpp & (tpp - 1)) == 0;
    if (d->c_out == 1 && d->c_in % 8 == 0 && pow2 && d->ntaps <= 9 && ((uintptr_t)in & 15) == 0) {
      long long need = (long long)d->n * d->grid_h, cap = (long long)ctx->num_sms * 8;   // one image row per block iteration
      int grid = (int)(need < cap ? need : cap);
      if (d->in_dt == SG_F32)
        sg_launch(ctx, k_conv_fwd_cout1<float>, grid, 256, 0, *d, (const float*)in, w_master, bias, mask, out);
      else
        sg_launch(ctx, k_conv_fwd_cout1<__nv_bfloat16>, grid, 256, 0, *d, (const __nv_bfloat16*)in, w_master, bias, mask, out);
      SG_POST_LAUNCH(ctx);
      return SG_OK;
    }
  }
  {
    bool unit = d->in_sy == 1 && d->in_sx == 1 && d->out_sy == 1 && d->out_sx == 1 && d->out_py == 0 && d->out_px == 0;
    int groups = d->c_out / 8;
    bool g_ok = d->c_out % 8 == 0 && groups >= 1 && groups <= 32 && 256 % groups == 0;
    if (unit && d->c_in == 1 && g_ok && d->ntaps <= 9 && d->in_dt == SG_F32 && !mask && ((uintptr_t)out & 15) == 0 && M < (1LL << 30)) {
      const bool wide = d->c_out % 32 == 0 && 256 % (d->c_out / 32) == 0;
      const int ppb = 256 / (wide ? d->c_out / 32 : groups);
      long long need = (M + ppb - 1) / ppb, cap = (long long)ctx->num_sms * 10;
      int grid = (int)(need < cap ? need : cap);
      if (wide) {
        if (d->out_dt == SG_F32) sg_launch(ctx, k_conv_fwd_cin1<float, 32>, grid, 256, 0, *d, (const float*)in, w_master, bias, (float*)out);
        else sg_launch(ctx, k_conv_fwd_cin1<__nv_bfloat16, 32>, grid, 256, 0, *d, (const float*)in, w_master, bias, (__nv_bfloat16*)out);
      } else {
        if (d->out_dt == SG_F32) sg_launch(ctx, k_conv_fwd_cin1<float, 8>, grid, 256, 0, *d, (const float*)in, w_master, bias, (float*)out);
        else sg_launch(ctx, k_conv_fwd_cin1<__nv_bfloat16, 8>, grid, 256, 0, *d, (const float*)in, w_master, bias, (__nv_bfloat16*)out);
      }
      SG_POST_LAUNCH(ctx);
      return SG_OK;
    }
  }
  if (d->c_out > 16) {
    dim3 grid(sg_div_up(M, CS_TM), sg_div_up(d->c_out, 64));
    sg_launch(ctx, k_conv_fwd_simt<64, 4>, grid, 256, 0, *d, in, w_master, bias, mask, out);
  } else {
    dim3 grid(sg_div_up(M, CS_TM), 1);
    sg_launch(ctx, k_conv_fwd_simt<16, 1>, grid, 256, 0, *d, in, w_master, bias, mask, out);
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_conv_wgrad_simt(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master) {
  SG_REQUIRE(ctx && in && dy && dw_master, "sg_conv_wgrad_simt: NULL");
  int rc = check_desc(d, "sg_conv_wgrad_simt");
  if (rc != SG_OK) return rc;
  long long P = (long long)d->n * d->grid_h * d->grid_w;
  if (P == 0) return SG_OK;
  {
    bool unit = d->in_sy == 1 && d->in_sx == 1 && d->out_sy == 1 && d->out_sx == 1 && d->out_py == 0 && d->out_px == 0;
    bool narrow_in = d->c_in == 1 && d->c_out <= 256 && 256 % d->c_out == 0;
    bool narrow_out = d->c_out == 1 && d->c_in <= 256 && 256 % d->c_in == 0;
    if (unit && d->ntaps <= 9 && ((narrow_in && d->c_out == 64) || (narrow_out && d->c_in == 64))) {
      // wide side = 64 channels: shared-memory staged skinny GEMM over pixels
      const void* wide = narrow_in ? dy : in;
      const void* nar = narrow_in ? in : dy;
      int wide_dt = narrow_in ? d->out_dt : d->in_dt, nar_dt = narrow_in ? d->in_dt : d->out_dt;
      int H = narrow_in ? d->out_h : d->in_h, W = narrow_in ? d->out_w : d->in_w;
      int nH = narrow_in ? d->in_h : d->out_h, nW = narrow_in ? d->in_w : d->out_w;
      // the pixel loop runs over the WIDE tensor; for c_in == 1 that must be exactly the output grid
      if ((!narrow_in || (d->grid_h == d->out_h && d->grid_w == d->out_w)) && (narrow_in || (d->grid_h == d->out_h && d->grid_w == d->out_w)) &&
          ((uintptr_t)wide & 15) == 0) {
        long long Pw = (long long)d->n * H * W;
        EdgeTaps tp0, tp;
        if (nH == H && nW == W && edge_taps(d, &tp0) && ((uintptr_t)nar & 15) == 0) {
          // patch position of tap t in the narrow tensor: +tap for c_in == 1 (narrow = input), -tap for c_out == 1 (narrow = dy)
          for (int i = 0; i < 9; ++i) tp.slot[i] = narrow_in ? tp0.slot[i] : tp0.slot[8 - i];
          long long need = (Pw / 4 + 31) / 32, cap = (long long)ctx->num_sms * 2;
          int grid = (int)(need < cap ? need : cap);
          if (wide_dt == SG_F32)
            sg_launch(ctx, k_wgrad_edge_q4<float>, grid, 256, 0, (const float*)wide, nar, nar_dt, d->n, H, W, tp, *d, dw_master, narrow_in ? 1 : 0,
                      ctx->det_scratch, ctx->det_tickets);
          else
            sg_launch(ctx, k_wgrad_edge_q4<__nv_bfloat16>, grid, 256, 0, (const __nv_bfloat16*)wide, nar, nar_dt, d->n, H, W, tp, *d, dw_master,
                      narrow_in ? 1 : 0, ctx->det_scratch, ctx->det_tickets);
          SG_POST_LAUNCH(ctx);
          return SG_OK;
        }
        long long nchunks = (Pw + WN_PIX - 1) / WN_PIX;
        long long blocks = (long long)ctx->num_sms * 4;
        if (blocks > nchunks) blocks = nchunks;
        long long cpb = (nchunks + blocks - 1) / blocks;
        blocks = (nchunks + cpb - 1) / cpb;
        if (wide_dt == SG_F32)
          sg_launch(ctx, k_wgrad_narrow64<float>, (int)blocks, 192, 0, (const float*)wide, nar, nar_dt, d->n, H, W, nH, nW, d->ntaps, *d,
                                                                       narrow_in ? 1 : -1, dw_master, cpb, narrow_in ? 1 : 0,
                                                                       ctx->det_scratch, ctx->det_tickets);
        else
          sg_launch(ctx, k_wgrad_narrow64<__nv_bfloat16>, (int)blocks, 192, 0, (const __nv_bfloat16*)wide, nar, nar_dt, d->n, H, W, nH,
                                                                               nW, d->ntaps, *d, narrow_in ? 1 : -1, dw_master, cpb,
                                                                               narrow_in ? 1 : 0, ctx->det_scratch, ctx->det_tickets);
        SG_POST_LAUNCH(ctx);
        return SG_OK;
      }
    }
    if (unit && (narrow_in || narrow_out)) {
      int wide = narrow_in ? d->c_out : d->c_in;
      int lanes = 256 / wide;
      long long blocks = (long long)ctx->num_sms * 4;
      long long min_pos = 8LL * lanes;
      if (blocks > (P + min_pos - 1) / min_pos) blocks = (P + min_pos - 1) / min_pos;
      long long ppb = (P + blocks - 1) / blocks;
      blocks = (P + ppb - 1) / ppb;
      size_t smem = sizeof(float) * (size_t)lanes * d->ntaps * wide;
      if (narrow_in) sg_launch(ctx, k_wgrad_narrow<true>, (int)blocks, 256, smem, *d, in, dy, dw_master, ppb, ctx->det_scratch, ctx->det_tickets);
      else sg_launch(ctx, k_wgrad_narrow<false>, (int)blocks, 256, smem, *d, in, dy, dw_master, ppb, ctx->det_scratch, ctx->det_tickets);
      SG_POST_LAUNCH(ctx);
      return SG_OK;
    }
  }
  int gx = sg_div_up(d->ntaps * d->c_in, CS_TM), gy = sg_div_up(d->c_out, 64);
  long long tiles = (long long)gx * gy;
  long long splits = (2LL * ctx->num_sms + tiles - 1) / tiles;
  long long max_splits = (P + 255) / 256;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if (splits > 65535) splits = 65535;
  if (tiles > SG_DET_TICKETS) splits = 1;      // no turn semaphores for that many tiles: one block per tile
  long long pps = ((P + splits - 1) / splits + CS_TK - 1) / CS_TK * CS_TK;
  splits = (P + pps - 1) / pps;
  dim3 grid(gx, gy, (unsigned)splits);
  sg_launch(ctx, k_conv_wgrad_simt, grid, 256, 0, *d, in, dy, dw_master, pps, ctx->det_tickets);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
