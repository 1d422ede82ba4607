// 1x1 projections of the non-local (self-attention) block, forward and backward, fused per data-flow step.
// Reference: arch_ops.py:38-46,55-57 (theta / phi / g projections), :63-67 (output projection, sigma * o + x).
//
// All of these are skinny GEMMs over p = n*h*w pixel rows with K, N in {32, 48, 64}: HBM-bound (each operand should
// move once), far too narrow for a 128-wide tensor-core tile, so they are FFMA kernels that stream a tile of rows
// through shared memory:
//   k_nl_rowgemm<K,N>  C[p,N] (+)= alpha * A[p,K] . W[K,N]      block = 128 rows x 2 column halves, W resident in smem,
//                                                                A tile staged with coalesced float4 loads
//   k_nl_wgrad<KA,KB>  dW[KA,KB] += alpha * A[p,KA]^T . B[p,KB]  reduction over rows: each block owns a slab of rows,
//                                                                keeps a 4x4 register tile per thread and adds its
//                                                                partial dW with one atomicAdd per element
// A, B, C and W may be "column-segmented": the logical matrix is the concatenation of up to three separate row-major
// arrays (theta | phi | g), which is how the three projections are computed from ONE pass over x.
#include "common.cuh"

struct SegMat {
  float* p[3];
  int w[3];      // widths (multiples of 4); unused segments have w = 0
};

__device__ __forceinline__ void seg_find(const SegMat& m, int col, int& s, int& off) {
  s = 0;
  off = col;
  if (off >= m.w[0]) { off -= m.w[0]; s = 1; if (off >= m.w[1]) { off -= m.w[1]; s = 2; } }
}

// W logical [K,N]; if TRANS_W the stored matrix is the column-segmented [N, K] one and is read transposed.
// Thread tile 4 rows x 4 columns: per k one LDS.128 of the (transposed) A tile and one LDS.128 of W feed 16 FMAs;
// a warp's stores cover whole 256-byte rows of C.
template <int K, int N>
struct NlTile {
  static constexpr int NCG = N / 4;                 // column groups
  static constexpr int RG = 256 / NCG;              // row groups per block
  static constexpr int TR = 4 * RG;                 // rows per tile
  static constexpr int TRP = (TR + 31) / 32 * 32 + 4;   // == 4 (mod 32): conflict-free STS.128 of the transposed tile
};

template <int K, int N, bool TRANS_W>
__global__ void __launch_bounds__(256) k_nl_rowgemm(long long rows, SegMat A, SegMat W, SegMat C, const float* __restrict__ alpha_p,
                                                     int accumulate, const float* __restrict__ resid_scale_p,
                                                     const float* __restrict__ resid_x, float* __restrict__ resid_out) {
  using T = NlTile<K, N>;
  __shared__ __align__(16) float As[K][T::TRP];     // transposed: As[k][row]
  __shared__ __align__(16) float Ws[K][N];
  const int tid = threadIdx.x;
  for (int i = tid; i < K * N; i += 256) {
    int k = i / N, n = i % N;
    int s, off;
    float v;
    if (!TRANS_W) {            // stored [K, N] column-segmented over n
      seg_find(W, n, s, off);
      v = W.p[s][(long long)k * W.w[s] + off];
    } else {                   // stored [N, K] column-segmented over k
      seg_find(W, k, s, off);
      v = W.p[s][(long long)n * W.w[s] + off];
    }
    Ws[k][n] = v;
  }
  const float alpha = alpha_p ? *alpha_p : 1.f;
  const float rscale = resid_scale_p ? *resid_scale_p : 1.f;
  const int cg = tid % T::NCG, rg = tid / T::NCG;
  const bool active = rg < T::RG;

  for (long long row0 = (long long)blockIdx.x * T::TR; row0 < rows; row0 += (long long)gridDim.x * T::TR) {
    const int cnt = rows - row0 < T::TR ? (int)(rows - row0) : T::TR;
    __syncthreads();
    // ---- A tile -> smem, transposed: item = (row quad, k); 4 coalesced row reads -> one STS.128 ----
    int koff = 0;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int w = A.w[s];
      if (w == 0) continue;
      const float* src = A.p[s] + row0 * w;
      for (int i = tid; i < T::RG * w; i += 256) {
        const int kk = i % w, rq = i / w;
        float4 v;
        const int r = 4 * rq;
        v.x = r < cnt ? src[(long long)r * w + kk] : 0.f;
        v.y = r + 1 < cnt ? src[(long long)(r + 1) * w + kk] : 0.f;
        v.z = r + 2 < cnt ? src[(long long)(r + 2) * w + kk] : 0.f;
        v.w = r + 3 < cnt ? src[(long long)(r + 3) * w + kk] : 0.f;
        *reinterpret_cast<float4*>(&As[koff + kk][r]) = v;
      }
      koff += w;
    }
    __syncthreads();
    if (active && 4 * rg < cnt) {
      float acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 8
      for (int k = 0; k < K; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(&As[k][4 * rg]);
        const float4 b = *reinterpret_cast<const float4*>(&Ws[k][4 * cg]);
        acc[0][0] = fmaf(a.x, b.x, acc[0][0]); acc[0][1] = fmaf(a.x, b.y, acc[0][1]); acc[0][2] = fmaf(a.x, b.z, acc[0][2]); acc[0][3] = fmaf(a.x, b.w, acc[0][3]);
        acc[1][0] = fmaf(a.y, b.x, acc[1][0]); acc[1][1] = fmaf(a.y, b.y, acc[1][1]); acc[1][2] = fmaf(a.y, b.z, acc[1][2]); acc[1][3] = fmaf(a.y, b.w, acc[1][3]);
        acc[2][0] = fmaf(a.z, b.x, acc[2][0]); acc[2][1] = fmaf(a.z, b.y, acc[2][1]); acc[2][2] = fmaf(a.z, b.z, acc[2][2]); acc[2][3] = fmaf(a.z, b.w, acc[2][3]);
        acc[3][0] = fmaf(a.w, b.x, acc[3][0]); acc[3][1] = fmaf(a.w, b.y, acc[3][1]); acc[3][2] = fmaf(a.w, b.z, acc[3][2]); acc[3][3] = fmaf(a.w, b.w, acc[3][3]);
      }
      int s, off;
      seg_find(C, 4 * cg, s, off);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (4 * rg + i < cnt) {
          const long long row = row0 + 4 * rg + i;
          float4 v = make_float4(alpha * acc[i][0], alpha * acc[i][1], alpha * acc[i][2], alpha * acc[i][3]);
          float* cp = C.p[s] + row * C.w[s] + off;
          if (accumulate) {
            float4 o = sg_ld4(cp);
            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
          }
          sg_st4(cp, v);
          if (resid_out) {     // second output: resid_out = rscale * C + x   (sigma * og + x, arch_ops.py:67)
            float4 x = sg_ld4(resid_x + row * N + 4 * cg);
            sg_st4(resid_out + row * N + 4 * cg, make_float4(fmaf(rscale, v.x, x.x), fmaf(rscale, v.y, x.y), fmaf(rscale, v.z, x.z),
                                                             fmaf(rscale, v.w, x.w)));
          }
        }
      }
    }
  }
}

// dW[KA,KB] += alpha * A^T . B over rows.  A block is SUB sub-blocks of (KA/4)*(KB/4) threads; every sub-block streams its
// own 32-row chunks through its own shared-memory buffers (more warps per SM to hide the load -> sync -> FMA latency
// chain), the sub-block partials are combined through shared memory and the block issues ONE atomicAdd per element.
#define NLW_ROWS 32
#define NLW_SUB 4
template <int KA, int KB>
__global__ void __launch_bounds__(NLW_SUB * (KA / 4) * (KB / 4)) k_nl_wgrad(long long rows, long long rows_per_block, SegMat A, SegMat B,
                                                                             SegMat DW, const float* __restrict__ alpha_p,
                                                                             float* __restrict__ scratch, unsigned int* __restrict__ ticket) {
  constexpr int TA = KA / 4, TB = KB / 4, NT = TA * TB;
  extern __shared__ __align__(16) float nlw_smem[];
  const int sub = threadIdx.x / NT, tid = threadIdx.x % NT;
  float (*As)[KA] = reinterpret_cast<float (*)[KA]>(nlw_smem + (size_t)sub * NLW_ROWS * (KA + KB));
  float (*Bs)[KB] = reinterpret_cast<float (*)[KB]>(nlw_smem + (size_t)sub * NLW_ROWS * (KA + KB) + NLW_ROWS * KA);
  const int ti = tid % TA, tj = tid / TA;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  for (long long base = r0; base < r1; base += (long long)NLW_SUB * NLW_ROWS) {
    const long long row0 = base + (long long)sub * NLW_ROWS;
    int cnt = 0;
    if (row0 < r1) cnt = r1 - row0 < NLW_ROWS ? (int)(r1 - row0) : NLW_ROWS;
    __syncthreads();
    int koff = 0;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int w = A.w[s];
      if (w == 0) continue;
      const float4* src = reinterpret_cast<const float4*>(A.p[s] + row0 * w);
      for (int i = tid; i < cnt * w / 4; i += NT) {
        int e = i * 4, rr = e / w, cc = e % w + koff;
        *reinterpret_cast<float4*>(&As[rr][cc]) = src[i];
      }
      koff += w;
    }
    koff = 0;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int w = B.w[s];
      if (w == 0) continue;
      const float4* src = reinterpret_cast<const float4*>(B.p[s] + row0 * w);
      for (int i = tid; i < cnt * w / 4; i += NT) {
        int e = i * 4, rr = e / w, cc = e % w + koff;
        *reinterpret_cast<float4*>(&Bs[rr][cc]) = src[i];
      }
      koff += w;
    }
    __syncthreads();
#pragma unroll 4
    for (int rr = 0; rr < cnt; ++rr) {
      float4 a = *reinterpret_cast<const float4*>(&As[rr][4 * ti]);
      float4 b = *reinterpret_cast<const float4*>(&Bs[rr][4 * tj]);
      acc[0][0] = fmaf(a.x, b.x, acc[0][0]); acc[0][1] = fmaf(a.x, b.y, acc[0][1]); acc[0][2] = fmaf(a.x, b.z, acc[0][2]); acc[0][3] = fmaf(a.x, b.w, acc[0][3]);
      acc[1][0] = fmaf(a.y, b.x, acc[1][0]); acc[1][1] = fmaf(a.y, b.y, acc[1][1]); acc[1][2] = fmaf(a.y, b.z, acc[1][2]); acc[1][3] = fmaf(a.y, b.w, acc[1][3]);
      acc[2][0] = fmaf(a.z, b.x, acc[2][0]); acc[2][1] = fmaf(a.z, b.y, acc[2][1]); acc[2][2] = fmaf(a.z, b.z, acc[2][2]); acc[2][3] = fmaf(a.z, b.w, acc[2][3]);
      acc[3][0] = fmaf(a.w, b.x, acc[3][0]); acc[3][1] = fmaf(a.w, b.y, acc[3][1]); acc[3][2] = fmaf(a.w, b.z, acc[3][2]); acc[3][3] = fmaf(a.w, b.w, acc[3][3]);
    }
  }
  // combine the sub-block partials: red[sub][16][NT] (re-using the staging buffers; NLW_SUB*16*NT <= NLW_SUB*NLW_ROWS*(KA+KB))
  __syncthreads();
  float* red = nlw_smem;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) red[((size_t)sub * 16 + i * 4 + j) * NT + tid] = acc[i][j];
  __syncthreads();
  // deterministic combine across blocks (common.cuh, scheme B): the block's [KA][KB] partial goes to its scratch slot
  if (sub == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = acc[i][j];
#pragma unroll
        for (int u = 1; u < NLW_SUB; ++u) v += red[((size_t)u * 16 + i * 4 + j) * NT + tid];
        scratch[(long long)blockIdx.x * (KA * KB) + (4 * ti + i) * KB + 4 * tj + j] = v;
      }
    }
  }
  const float alpha = alpha_p ? *alpha_p : 1.f;
  sg_det_finish(scratch, scratch + (long long)gridDim.x * (KA * KB), ticket, gridDim.x, blockIdx.x, KA * KB, [&](int i, float sum) {
    int r = i / KB, c = i % KB, s, off;
    seg_find(DW, c, s, off);
    DW.p[s][(long long)r * DW.w[s] + off] += alpha * sum;
  });
}

// ---------------------------------------------------------------------------------------------------
// bf16 speed mode: the same two operations on warp-level tensor ops (mma.sync m16n8k16, fp32 accumulate).
// The FFMA kernels above are instruction bound (~2x the 64x48 FMAs per row in issue slots); here a warp owns 16 rows, loads
// the fp32 operands straight from global memory in fragment order (every 32-byte sector is used exactly once, no staging
// of the activations), converts to bf16 in registers, and the kernels become HBM bound.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t nl_pack(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void nl_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// C[rows,N] (+)= alpha * A[rows,K] . W[K,N]; 8 warps x 16 rows per block iteration; W^T (bf16) resident in smem
template <int K, int N, bool TRANS_W>
__global__ void __launch_bounds__(256) k_nl_rowgemm_mma(long long rows, SegMat A, SegMat W, SegMat C, const float* __restrict__ alpha_p,
                                                         int accumulate, const float* __restrict__ resid_scale_p,
                                                         const float* __restrict__ resid_x, float* __restrict__ resid_out) {
  constexpr int KP = K + 8;                                  // padded row (bf16): conflict-free 32-bit fragment reads
  __shared__ __align__(16) __nv_bfloat16 Wt[N * KP];         // Wt[n][k] = Wlogical[k][n]
  for (int i = threadIdx.x; i < K * N; i += 256) {
    int k = i / N, n = i % N;
    int s, off;
    float v;
    if (!TRANS_W) { seg_find(W, n, s, off); v = W.p[s][(long long)k * W.w[s] + off]; }
    else { seg_find(W, k, s, off); v = W.p[s][(long long)n * W.w[s] + off]; }
    Wt[n * KP + k] = __float2bfloat16_rn(v);
  }
  __syncthreads();
  const float alpha = alpha_p ? *alpha_p : 1.f;
  const float rscale = resid_scale_p ? *resid_scale_p : 1.f;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  for (long long r0 = ((long long)blockIdx.x * 8 + warp) * 16; r0 < rows; r0 += (long long)gridDim.x * 128) {
    const long long ra = r0 + g, rb = r0 + g + 8;
    const long long ca = ra < rows ? ra : rows - 1, cb = rb < rows ? rb : rows - 1;
    uint32_t a[K / 16][4];
#pragma unroll
    for (int ks = 0; ks < K / 16; ++ks) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {                          // k halves of 8 never straddle a segment (widths % 8 == 0)
        int s, off;
        seg_find(A, 16 * ks + 8 * h, s, off);
        const float2 va = *reinterpret_cast<const float2*>(A.p[s] + ca * A.w[s] + off + 2 * t);
        const float2 vb = *reinterpret_cast<const float2*>(A.p[s] + cb * A.w[s] + off + 2 * t);
        a[ks][2 * h] = nl_pack(va.x, va.y);
        a[ks][2 * h + 1] = nl_pack(vb.x, vb.y);
      }
    }
#pragma unroll
    for (int nt = 0; nt < N / 8; ++nt) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < K / 16; ++ks) {
        const __nv_bfloat16* wp = Wt + (8 * nt + g) * KP + 16 * ks + 2 * t;
        nl_mma(acc, a[ks], *reinterpret_cast<const uint32_t*>(wp), *reinterpret_cast<const uint32_t*>(wp + 8));
      }
      int s, off;
      seg_find(C, 8 * nt, s, off);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const long long row = h ? rb : ra;
        if (row >= rows) continue;
        float2 v = make_float2(alpha * acc[2 * h], alpha * acc[2 * h + 1]);
        float* cp = C.p[s] + row * C.w[s] + off + 2 * t;
        if (accumulate) {
          float2 o = *reinterpret_cast<const float2*>(cp);
          v.x += o.x; v.y += o.y;
        }
        *reinterpret_cast<float2*>(cp) = v;
        if (resid_out) {
          const float2 x = *reinterpret_cast<const float2*>(resid_x + row * N + 8 * nt + 2 * t);
          *reinterpret_cast<float2*>(resid_out + row * N + 8 * nt + 2 * t) = make_float2(fmaf(rscale, v.x, x.x), fmaf(rscale, v.y, x.y));
        }
      }
    }
  }
}

// dW[KA,KB] += alpha * A^T . B over rows: a warp keeps the WHOLE dW tile in accumulator fragments ((KA/16) x (KB/8) mma
// tiles) and walks 16-row chunks; A^T and B fragments are pairs of consecutive ROWS of one column, read straight from
// global memory (8 lanes cover one 32-byte sector).  The 8 warps of a block are combined with shared-memory atomics,
// then one global atomicAdd per element and block.
template <int KA, int KB>
__global__ void __launch_bounds__(256, 1) k_nl_wgrad_mma(long long rows, long long rows_per_block, SegMat A, SegMat B, SegMat DW,
                                                          const float* __restrict__ alpha_p, float* __restrict__ scratch,
                                                          unsigned int* __restrict__ ticket) {
  constexpr int MT = KA / 16, NT = KB / 8;
  __shared__ float red[KA * KB];
  for (int i = threadIdx.x; i < KA * KB; i += 256) red[i] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  float acc[MT][NT][4];
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n) acc[m][n][0] = acc[m][n][1] = acc[m][n][2] = acc[m][n][3] = 0.f;
  long long r_begin = (long long)blockIdx.x * rows_per_block, r_end = r_begin + rows_per_block;
  if (r_end > rows) r_end = rows;
  for (long long r0 = r_begin + warp * 16; r0 < r_end; r0 += 128) {
    // the four row pairs of this chunk that this lane touches: rows 2t, 2t+1, 2t+8, 2t+9 (zero beyond r_end)
    long long rr[4] = {r0 + 2 * t, r0 + 2 * t + 1, r0 + 2 * t + 8, r0 + 2 * t + 9};
    bool ok[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { ok[i] = rr[i] < r_end; if (!ok[i]) rr[i] = r_end - 1; }
    uint32_t af[MT][4];
#pragma unroll
    for (int m = 0; m < MT; ++m) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {                          // column 16m + g + 8h of A
        int s, off;
        seg_find(A, 16 * m + 8 * h, s, off);
        const float* base = A.p[s] + off + g;
        const long long w = A.w[s];
        float v0 = ok[0] ? base[rr[0] * w] : 0.f, v1 = ok[1] ? base[rr[1] * w] : 0.f;
        float v2 = ok[2] ? base[rr[2] * w] : 0.f, v3 = ok[3] ? base[rr[3] * w] : 0.f;
        af[m][h] = nl_pack(v0, v1);                          // a0 / a1: k = rows 2t, 2t+1
        af[m][2 + h] = nl_pack(v2, v3);                      // a2 / a3: k = rows 2t+8, 2t+9
      }
    }
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      int s, off;
      seg_find(B, 8 * n, s, off);
      const float* base = B.p[s] + off + g;
      const long long w = B.w[s];
      float v0 = ok[0] ? base[rr[0] * w] : 0.f, v1 = ok[1] ? base[rr[1] * w] : 0.f;
      float v2 = ok[2] ? base[rr[2] * w] : 0.f, v3 = ok[3] ? base[rr[3] * w] : 0.f;
      const uint32_t b0 = nl_pack(v0, v1), b1 = nl_pack(v2, v3);
#pragma unroll
      for (int m = 0; m < MT; ++m) nl_mma(acc[m][n], af[m], b0, b1);
    }
  }
  // accumulator (m tile, n tile): c0,c1 = (row 16m + g, cols 8n + 2t, +1); c2,c3 = row + 8.  The 8 warps add their
  // fragments into the block tile one warp after the other (fixed order: bitwise repeatable), then the blocks are combined
  // in block order by the last block to arrive (common.cuh, scheme B)
  for (int w = 0; w < 8; ++w) {
    if (warp == w) {
#pragma unroll
      for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int n = 0; n < NT; ++n) {
          red[(16 * m + g) * KB + 8 * n + 2 * t] += acc[m][n][0];
          red[(16 * m + g) * KB + 8 * n + 2 * t + 1] += acc[m][n][1];
          red[(16 * m + g + 8) * KB + 8 * n + 2 * t] += acc[m][n][2];
          red[(16 * m + g + 8) * KB + 8 * n + 2 * t + 1] += acc[m][n][3];
        }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < KA * KB; i += 256) scratch[(long long)blockIdx.x * (KA * KB) + i] = red[i];
  const float alpha = alpha_p ? *alpha_p : 1.f;
  sg_det_finish(scratch, scratch + (long long)gridDim.x * (KA * KB), ticket, gridDim.x, blockIdx.x, KA * KB, [&](int i, float sum) {
    int r = i / KB, c = i % KB, s, off;
    seg_find(DW, c, s, off);
    DW.p[s][(long long)r * DW.w[s] + off] += alpha * sum;
  });
}

template <int K, int N, bool TRANS_W>
static int nl_rowgemm_launch(sg_ctx* ctx, long long rows, SegMat A, SegMat W, SegMat C, const float* alpha, int accumulate,
                             const float* resid_scale, const float* resid_x, float* resid_out);

static SegMat seg1(const float* a, int w) {
  SegMat m;
  m.p[0] = const_cast<float*>(a); m.p[1] = m.p[2] = nullptr;
  m.w[0] = w; m.w[1] = m.w[2] = 0;
  return m;
}
static SegMat seg3(const float* a, int wa, const float* b, int wb, const float* c, int wc) {
  SegMat m;
  m.p[0] = const_cast<float*>(a); m.p[1] = const_cast<float*>(b); m.p[2] = const_cast<float*>(c);
  m.w[0] = wa; m.w[1] = wb; m.w[2] = wc;
  return m;
}
template <int K, int N>
static int nl_grid(sg_ctx* ctx, long long rows) {
  long long need = (rows + NlTile<K, N>::TR - 1) / NlTile<K, N>::TR, cap = (long long)ctx->num_sms * 6;
  return (int)(need < cap ? need : cap);
}
static void nl_wgrad_grid(sg_ctx* ctx, long long rows, int* grid, long long* rpb) {
  long long blocks = (long long)ctx->num_sms * 2;
  const long long step = (long long)NLW_SUB * NLW_ROWS;
  long long r = (rows + blocks - 1) / blocks;
  r = (r + step - 1) / step * step;
  *rpb = r;
  *grid = (int)((rows + r - 1) / r);
}
template <int KA, int KB>
static int nl_wgrad_launch(sg_ctx* ctx, long long rows, SegMat A, SegMat B, SegMat DW, const float* alpha) {
  if (ctx->speed_mode) {
    long long blocks = (long long)ctx->num_sms * 2;
    long long rpb = ((rows + blocks - 1) / blocks + 127) / 128 * 128;
    int grid_m = (int)((rows + rpb - 1) / rpb);
    sg_launch(ctx, k_nl_wgrad_mma<KA, KB>, grid_m, 256, 0, rows, rpb, A, B, DW, alpha, ctx->det_scratch, ctx->det_tickets);
    SG_POST_LAUNCH(ctx);
    return SG_OK;
  }
  int grid;
  long long rpb;
  nl_wgrad_grid(ctx, rows, &grid, &rpb);
  size_t smem = sizeof(float) * (size_t)NLW_SUB * NLW_ROWS * (KA + KB);
  static_assert(NLW_SUB * 16 * (KA / 4) * (KB / 4) <= NLW_SUB * NLW_ROWS * (KA + KB), "reduction buffer does not fit");
  SG_CHECK_CUDA(cudaFuncSetAttribute(k_nl_wgrad<KA, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  sg_launch(ctx, k_nl_wgrad<KA, KB>, grid, NLW_SUB * (KA / 4) * (KB / 4), smem, rows, rpb, A, B, DW, alpha, ctx->det_scratch,
                                                                                  ctx->det_tickets);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

template <int K, int N, bool TRANS_W>
static int nl_rowgemm_launch(sg_ctx* ctx, long long rows, SegMat A, SegMat W, SegMat C, const float* alpha, int accumulate,
                             const float* resid_scale, const float* resid_x, float* resid_out) {
  if (ctx->speed_mode) {
    long long need = (rows + 127) / 128, cap = (long long)ctx->num_sms * 8;
    sg_launch(ctx, k_nl_rowgemm_mma<K, N, TRANS_W>, (int)(need < cap ? need : cap), 256, 0, rows, A, W, C, alpha, accumulate, resid_scale,
                                                                                            resid_x, resid_out);
  } else {
    sg_launch(ctx, k_nl_rowgemm<K, N, TRANS_W>, nl_grid<K, N>(ctx, rows), 256, 0, rows, A, W, C, alpha, accumulate, resid_scale, resid_x,
                                                                                  resid_out);
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

#define NL_C 64
#define NL_DK 8
#define NL_DV 32
#define NL_ALIGNED(p) ((((uintptr_t)(p)) & 15) == 0)

extern "C" {

int sg_nonlocal_proj_fwd(sg_ctx* ctx, const float* x, long long rows, const float* w_theta, const float* w_phi,
                         const float* w_g, float* theta, float* phi_f, float* g_f) {
  SG_REQUIRE(ctx && x && w_theta && w_phi && w_g && theta && phi_f && g_f, "sg_nonlocal_proj_fwd: NULL");
  SG_REQUIRE(NL_ALIGNED(x) && NL_ALIGNED(theta) && NL_ALIGNED(phi_f) && NL_ALIGNED(g_f), "sg_nonlocal_proj_fwd: 16-byte alignment");
  if (rows == 0) return SG_OK;
  return nl_rowgemm_launch<NL_C, 2 * NL_DK + NL_DV, false>(ctx, rows, seg1(x, NL_C), seg3(w_theta, NL_DK, w_phi, NL_DK, w_g, NL_DV),
                                                           seg3(theta, NL_DK, phi_f, NL_DK, g_f, NL_DV), nullptr, 0, nullptr, nullptr, nullptr);
}

int sg_nonlocal_out_fwd(sg_ctx* ctx, const float* o, long long rows, const float* w_o, const float* sigma, const float* x,
                        float* og, float* out) {
  SG_REQUIRE(ctx && o && w_o && sigma && x && og && out, "sg_nonlocal_out_fwd: NULL");
  SG_REQUIRE(NL_ALIGNED(o) && NL_ALIGNED(x) && NL_ALIGNED(og) && NL_ALIGNED(out), "sg_nonlocal_out_fwd: 16-byte alignment");
  if (rows == 0) return SG_OK;
  // og = o . Wo (kept un-scaled for d sigma = <dout, og>);  out = sigma * og + x
  return nl_rowgemm_launch<NL_DV, NL_C, false>(ctx, rows, seg1(o, NL_DV), seg1(w_o, NL_C), seg1(og, NL_C), nullptr, 0, sigma, x, out);
}

int sg_nonlocal_out_bwd(sg_ctx* ctx, const float* dout, const float* o, long long rows, const float* w_o, const float* sigma,
                        float* d_o, float* dw_o) {
  SG_REQUIRE(ctx && dout && o && w_o && sigma && d_o, "sg_nonlocal_out_bwd: NULL");
  SG_REQUIRE(NL_ALIGNED(dout) && NL_ALIGNED(o) && NL_ALIGNED(d_o), "sg_nonlocal_out_bwd: 16-byte alignment");
  if (rows == 0) return SG_OK;
  // d_o = sigma * dout . Wo^T
  int rc = nl_rowgemm_launch<NL_C, NL_DV, true>(ctx, rows, seg1(dout, NL_C), seg1(w_o, NL_C), seg1(d_o, NL_DV), sigma, 0, nullptr, nullptr,
                                                nullptr);
  if (rc != SG_OK) return rc;
  if (dw_o)                    // dWo[32,64] += sigma * o^T . dout
    return nl_wgrad_launch<NL_DV, NL_C>(ctx, rows, seg1(o, NL_DV), seg1(dout, NL_C), seg1(dw_o, NL_C), sigma);
  return SG_OK;
}

int sg_nonlocal_proj_bwd(sg_ctx* ctx, const float* x, const float* dtheta, const float* dphi_f, const float* dg_f, long long rows,
                         const float* w_theta, const float* w_phi, const float* w_g, float* dx, float* dw_theta, float* dw_phi,
                         float* dw_g) {
  SG_REQUIRE(ctx && x && dtheta && dphi_f && dg_f && w_theta && w_phi && w_g && dx, "sg_nonlocal_proj_bwd: NULL");
  SG_REQUIRE(NL_ALIGNED(x) && NL_ALIGNED(dtheta) && NL_ALIGNED(dphi_f) && NL_ALIGNED(dg_f) && NL_ALIGNED(dx),
             "sg_nonlocal_proj_bwd: 16-byte alignment");
  SG_REQUIRE((dw_theta != nullptr) == (dw_phi != nullptr) && (dw_phi != nullptr) == (dw_g != nullptr),
             "sg_nonlocal_proj_bwd: give all three filter gradients or none");
  if (rows == 0) return SG_OK;
  SegMat d = seg3(dtheta, NL_DK, dphi_f, NL_DK, dg_f, NL_DV);
  // dx += [dtheta | dphi | dg] . [Wtheta | Wphi | Wg]^T
  int rc = nl_rowgemm_launch<2 * NL_DK + NL_DV, NL_C, true>(ctx, rows, d, seg3(w_theta, NL_DK, w_phi, NL_DK, w_g, NL_DV), seg1(dx, NL_C), nullptr,
                                                            1, nullptr, nullptr, nullptr);
  if (rc != SG_OK) return rc;
  if (dw_theta)                // [dWtheta | dWphi | dWg] += x^T . [dtheta | dphi | dg]
    return nl_wgrad_launch<NL_C, 2 * NL_DK + NL_DV>(ctx, rows, seg1(x, NL_C), d, seg3(dw_theta, NL_DK, dw_phi, NL_DK, dw_g, NL_DV), nullptr);
  return SG_OK;
}

}  // extern "C"
