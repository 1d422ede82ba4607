// Element-wise glue and pooling kernels: HBM-bound, float4-vectorised grid-stride loops,
// grids sized as a multiple of the SM count.
#include "common.cuh"

static inline int ew_grid(sg_ctx* ctx, long long work_items, int threads) {
  long long need = (work_items + threads - 1) / threads;
  long long cap = (long long)ctx->num_sms * 8;
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}

// ---------------------------------------------------------------------------------------------------
template <typename TO>
__global__ void k_act_prep(const float* __restrict__ x, long long n4, long long n, TO* __restrict__ relu_out,
                           TO* __restrict__ copy_out) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = sg_ld4(x + 4 * i);
    if (copy_out) sg_st4(copy_out + 4 * i, v);
    if (relu_out) sg_st4(relu_out + 4 * i, make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f)));
  }
  // tail
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = x[i];
    if (copy_out) sg_st(copy_out + i, v);
    if (relu_out) sg_st(relu_out + i, fmaxf(v, 0.f));
  }
}

template <typename TA, typename TO>
__global__ void k_mask_mul(const float* __restrict__ dy, const TA* __restrict__ act, TO* __restrict__ out,
                           long long n4, long long n, int accumulate) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 d = sg_ld4(dy + 4 * i);
    float4 a = sg_ld4(act + 4 * i);
    float4 r = make_float4(a.x > 0.f ? d.x : 0.f, a.y > 0.f ? d.y : 0.f, a.z > 0.f ? d.z : 0.f, a.w > 0.f ? d.w : 0.f);
    if (accumulate) {
      float4 o = sg_ld4(out + 4 * i);
      r.x += o.x; r.y += o.y; r.z += o.z; r.w += o.w;
    }
    sg_st4(out + 4 * i, r);
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float r = sg_ld(act + i) > 0.f ? dy[i] : 0.f;
    if (accumulate) r += sg_ld(out + i);
    sg_st(out + i, r);
  }
}

__global__ void k_axpby(float a, const float* __restrict__ x, float b, const float* __restrict__ y,
                        float* __restrict__ out, long long n4, long long n) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = sg_ld4(x + 4 * i);
    float4 r = make_float4(a * v.x, a * v.y, a * v.z, a * v.w);
    if (y) {
      float4 w = sg_ld4(y + 4 * i);
      r.x += b * w.x; r.y += b * w.y; r.z += b * w.z; r.w += b * w.w;
    }
    sg_st4(out + 4 * i, r);
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float r = a * x[i];
    if (y) r += b * y[i];
    out[i] = r;
  }
}

__global__ void k_scale_add(const float* __restrict__ sigma, const float* __restrict__ a,
                            const float* __restrict__ x, float* __restrict__ out, long long n4, long long n) {
  const float s = *sigma;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = sg_ld4(a + 4 * i), w = x ? sg_ld4(x + 4 * i) : make_float4(0, 0, 0, 0);
    sg_st4(out + 4 * i, make_float4(s * v.x + w.x, s * v.y + w.y, s * v.z + w.z, s * v.w + w.w));
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = s * a[i] + (x ? x[i] : 0.f);
}

__global__ void k_tanh_fwd(const float* __restrict__ x, float* __restrict__ y, long long n) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] = tanhf(x[i]);
}
__global__ void k_tanh_bwd(const float* __restrict__ dy, const float* __restrict__ y, float* __restrict__ dx,
                           long long n) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float t = y[i];
    dx[i] = dy[i] * (1.f - t * t);
  }
}
__global__ void k_scale_rows(float* __restrict__ x, const float* __restrict__ w, int rows, long long cols) {
  long long n = (long long)rows * cols;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] *= w[i / cols];
}

// x[i, :] *= up[i] * mult for the samples i of a batch-first tensor (8 elements per thread; per_sample % 8 == 0).  Samples whose
// factor is exactly 1 are left alone and samples whose factor is 0 are only written: with the hinge loss the factors of the
// merged discriminator backward (net_architecture.py: Discriminator.backward_merged) are exactly those two values.
// grid: (blocks per sample, samples)
template <typename T>
__global__ void __launch_bounds__(256) k_scale_samples(T* __restrict__ x, long long per_sample8, const float* __restrict__ up, float mult) {
  const float f = up[blockIdx.y] * mult;
  if (f == 1.0f) return;
  T* xs = x + (long long)blockIdx.y * per_sample8 * 8;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_sample8; i += stride) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (f != 0.0f) {
      a = sg_ld4(xs + 8 * i); b = sg_ld4(xs + 8 * i + 4);
      a.x *= f; a.y *= f; a.z *= f; a.w *= f; b.x *= f; b.y *= f; b.z *= f; b.w *= f;
    }
    sg_st4(xs + 8 * i, a); sg_st4(xs + 8 * i + 4, b);
  }
}

// deterministic: per-block partials, summed in block order by the block that arrives last (common.cuh, scheme B)
__global__ void k_dot(const float* __restrict__ a, const float* __restrict__ b, long long n, float* out, int accumulate,
                      float* __restrict__ scratch, unsigned int* ticket) {
  __shared__ float sm[32];
  float acc = 0.f;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) acc += a[i] * b[i];
  float t = sg_block_sum(acc, sm);
  if (threadIdx.x == 0) scratch[blockIdx.x] = t;
  if (!sg_det_arrive_last(ticket, gridDim.x)) return;
  float part = 0.f;
  for (unsigned int i = threadIdx.x; i < gridDim.x; i += blockDim.x) part += __ldcg(scratch + i);
  float tot = sg_block_sum(part, sm);
  if (threadIdx.x == 0) *out = (accumulate ? *out : 0.f) + tot;
}

// column sums of a [rows, cols] matrix (bias gradients): a block owns a slab of rows; its 256 threads are arranged as
// (cols/4 column groups) x (row lanes), every thread streams 4 adjacent columns with one 8/16-byte load per row, the
// row lanes are combined through shared memory and the block adds its partial sums with one atomicAdd per column.
template <typename T, int NT>
__global__ void __launch_bounds__(NT) k_colsum_v4(const T* __restrict__ x, long long rows, int cols, long long rows_per_block,
                                                    float* __restrict__ out, int accumulate, float* __restrict__ scratch,
                                                    unsigned int* ticket) {
  __shared__ float4 sm[NT];
  const int cgs = cols >> 2;                          // column groups of 4
  const int cg_per_pass = cgs < NT ? cgs : NT;
  const int lanes_r = NT / cg_per_pass;              // row lanes (>= 1)
  const int cgi = threadIdx.x % cg_per_pass, rl = threadIdx.x / cg_per_pass;
  long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  for (int cg0 = 0; cg0 < cgs; cg0 += cg_per_pass) {
    const int cg = cg0 + cgi;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rl < lanes_r && cg < cgs) {
      const T* p = x + (long long)cg * 4;
      long long r = r0 + rl;
      for (; r + 3LL * lanes_r < r1; r += 4LL * lanes_r) {
        float4 a = sg_ld4(p + r * cols), b = sg_ld4(p + (r + lanes_r) * cols), c = sg_ld4(p + (r + 2LL * lanes_r) * cols),
               d = sg_ld4(p + (r + 3LL * lanes_r) * cols);
        acc.x += (a.x + b.x) + (c.x + d.x); acc.y += (a.y + b.y) + (c.y + d.y);
        acc.z += (a.z + b.z) + (c.z + d.z); acc.w += (a.w + b.w) + (c.w + d.w);
      }
      for (; r < r1; r += lanes_r) {
        float4 a = sg_ld4(p + r * cols);
        acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
      }
    }
    __syncthreads();
    sm[threadIdx.x] = acc;
    __syncthreads();
    if (rl == 0 && cg < cgs) {
      for (int j = 1; j < lanes_r; ++j) {
        float4 o = sm[j * cg_per_pass + cgi];
        acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
      }
      if (gridDim.x == 1) {
        float* op = out + (long long)cg * 4;
        float4 prev = accumulate ? sg_ld4(op) : make_float4(0.f, 0.f, 0.f, 0.f);
        sg_st4(op, make_float4(prev.x + acc.x, prev.y + acc.y, prev.z + acc.z, prev.w + acc.w));
      } else {
        sg_st4(scratch + (long long)blockIdx.x * cols + (long long)cg * 4, acc);
      }
    }
  }
  if (gridDim.x == 1) return;
  // deterministic combine (common.cuh, scheme B): the last block to arrive sums the per-block partials in block order
  sg_det_finish(scratch, scratch + (long long)gridDim.x * cols, ticket, gridDim.x, blockIdx.x, cols,
                [&](int c, float t) { out[c] = (accumulate ? out[c] : 0.f) + t; });
}

// generic fallback (cols not a multiple of 4): thread t handles columns t, t+blockDim...
template <typename T>
__global__ void k_colsum(const T* __restrict__ x, long long rows, int cols, long long rows_per_block,
                         float* __restrict__ out, int accumulate, float* __restrict__ scratch, unsigned int* ticket) {
  long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float acc = 0.f;
    for (long long r = r0; r < r1; ++r) acc += sg_ld(x + r * cols + c);
    scratch[(long long)blockIdx.x * cols + c] = acc;
  }
  sg_det_finish(scratch, scratch + (long long)gridDim.x * cols, ticket, gridDim.x, blockIdx.x, cols,
                [&](int c, float t) { out[c] = (accumulate ? out[c] : 0.f) + t; });
}

template <typename TO>
__global__ void k_cast(const float* __restrict__ x, TO* __restrict__ out, long long n) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) sg_st(out + i, x[i]);
}

// ---------------------------------------------------------------------------------------------------
// pooling (NHWC, c % 4 == 0)
// ---------------------------------------------------------------------------------------------------
__global__ void k_avgpool2_fwd(const float* __restrict__ x, int n, int h, int w, int c4, float* __restrict__ out) {
  int ho = h / 2, wo = w / 2;
  long long total = (long long)n * ho * wo * c4;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int cc = (int)(i % c4);
    long long p = i / c4;
    int ox = (int)(p % wo);
    p /= wo;
    int oy = (int)(p % ho);
    int ni = (int)(p / ho);
    const float* base = x + (((long long)ni * h + 2 * oy) * w + 2 * ox) * (4LL * c4) + 4 * cc;
    float4 a = sg_ld4(base), b = sg_ld4(base + 4LL * c4), cq = sg_ld4(base + (long long)w * 4 * c4),
           d = sg_ld4(base + (long long)w * 4 * c4 + 4LL * c4);
    sg_st4(out + 4 * i, make_float4(0.25f * (a.x + b.x + cq.x + d.x), 0.25f * (a.y + b.y + cq.y + d.y),
                                    0.25f * (a.z + b.z + cq.z + d.z), 0.25f * (a.w + b.w + cq.w + d.w)));
  }
}

// one thread per (output-row pair, x pair, 4 channels): reads one float4 of dout, writes the 2 x 2 window (32-bit index
// math: one division chain per 4 stores instead of per store)
template <typename TO>
__global__ void k_avgpool2_bwd(const float* __restrict__ dout, int n, int h, int w, int c4, TO* __restrict__ dx) {
  const int ho = h / 2, wo = w / 2;
  const long long total = (long long)n * ho * wo * c4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long row_e = (long long)w * c4 * 4;       // elements per input row
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int cc = (int)(i % c4);
    const long long p = i / c4;                         // (ni*ho + oy)*wo + ox
    const int ox = (int)(p % wo);
    const long long r = p / wo;                         // ni*ho + oy  ->  input row 2*r (h = 2*ho)
    float4 v = sg_ld4(dout + 4 * i);
    v = make_float4(0.25f * v.x, 0.25f * v.y, 0.25f * v.z, 0.25f * v.w);
    TO* o = dx + 2 * r * row_e + ((long long)(2 * ox) * c4 + cc) * 4;
    sg_st4(o, v);
    sg_st4(o + 4LL * c4, v);
    sg_st4(o + row_e, v);
    sg_st4(o + row_e + 4LL * c4, v);
  }
}

template <typename T>
__global__ void k_maxpool_fwd(const T* __restrict__ x, int n, int h, int w, int c, int ph, int pw,
                              T* __restrict__ out) {
  int ho = h / ph, wo = w / pw;
  long long total = (long long)n * ho * wo * c;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int cc = (int)(i % c);
    long long p = i / c;
    int ox = (int)(p % wo);
    p /= wo;
    int oy = (int)(p % ho);
    int ni = (int)(p / ho);
    float m = -INFINITY;
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b)
        m = fmaxf(m, sg_ld(x + (((long long)ni * h + oy * ph + a) * w + ox * pw + b) * c + cc));
    sg_st(out + i, m);
  }
}

// 4 channels per thread (c % 4 == 0): 8/16-byte loads and stores
template <typename T>
__global__ void k_maxpool_fwd_v4(const T* __restrict__ x, int n, int h, int w, int c4, int ph, int pw, T* __restrict__ out) {
  int ho = h / ph, wo = w / pw;
  long long total = (long long)n * ho * wo * c4;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int cc = (int)(i % c4);
    long long p = i / c4;
    int ox = (int)(p % wo);
    p /= wo;
    int oy = (int)(p % ho);
    int ni = (int)(p / ho);
    float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b) {
        float4 v = sg_ld4(x + ((((long long)ni * h + oy * ph + a) * w + ox * pw + b) * c4 + cc) * 4);
        m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
      }
    sg_st4(out + 4 * i, m);
  }
}

template <typename TX, typename TO>
__global__ void k_maxpool_bwd_v4(const float* __restrict__ dout, const TX* __restrict__ x, int n, int h, int w, int c4,
                                 int ph, int pw, int relu_mask, TO* __restrict__ dx) {
  int ho = h / ph, wo = w / pw;
  long long total = (long long)n * ho * wo * c4;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int cc = (int)(i % c4);
    long long p = i / c4;
    int ox = (int)(p % wo);
    p /= wo;
    int oy = (int)(p % ho);
    int ni = (int)(p / ho);
    float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    int best[4] = {0, 0, 0, 0};
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b) {
        float4 v4 = sg_ld4(x + ((((long long)ni * h + oy * ph + a) * w + ox * pw + b) * c4 + cc) * 4);
        float v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (v[j] > m[j]) { m[j] = v[j]; best[j] = a * pw + b; }
      }
    float4 g4 = sg_ld4(dout + 4 * i);
    float g[4] = {g4.x, g4.y, g4.z, g4.w};
    if (relu_mask) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (!(m[j] > 0.f)) g[j] = 0.f;
    }
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b) {
        int k = a * pw + b;
        sg_st4(dx + ((((long long)ni * h + oy * ph + a) * w + ox * pw + b) * c4 + cc) * 4,
               make_float4(k == best[0] ? g[0] : 0.f, k == best[1] ? g[1] : 0.f, k == best[2] ? g[2] : 0.f, k == best[3] ? g[3] : 0.f));
      }
  }
}

// gradient goes to the FIRST maximal element of the window (row-major window order), optionally gated by x > 0
template <typename TX, typename TO>
__global__ void k_maxpool_bwd(const float* __restrict__ dout, const TX* __restrict__ x, int n, int h, int w, int c,
                              int ph, int pw, int relu_mask, TO* __restrict__ dx) {
  int ho = h / ph, wo = w / pw;
  long long total = (long long)n * ho * wo * c;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int cc = (int)(i % c);
    long long p = i / c;
    int ox = (int)(p % wo);
    p /= wo;
    int oy = (int)(p % ho);
    int ni = (int)(p / ho);
    float m = -INFINITY;
    int best = 0;
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b) {
        float v = sg_ld(x + (((long long)ni * h + oy * ph + a) * w + ox * pw + b) * c + cc);
        if (v > m) { m = v; best = a * pw + b; }
      }
    float g = dout[i];
    if (relu_mask && !(m > 0.f)) g = 0.f;
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b)
        sg_st(dx + (((long long)ni * h + oy * ph + a) * w + ox * pw + b) * c + cc, (a * pw + b == best) ? g : 0.f);
  }
}

// global average pool of relu(x): one block per (image, 128-channel slab); threads split (pixel-slices x channels)
__global__ void k_gap_relu_fwd(const float* __restrict__ x, long long hw, int c, float* __restrict__ out) {
  __shared__ float sm[8][128];
  int ni = blockIdx.y;
  int c0 = blockIdx.x * 128;
  int cl = threadIdx.x & 127, slice = threadIdx.x >> 7;     // 1024 threads: 8 slices
  int cc = c0 + cl;
  float acc = 0.f;
  if (cc < c)
    for (long long p = slice; p < hw; p += 8) acc += fmaxf(x[((long long)ni * hw + p) * c + cc], 0.f);
  sm[slice][cl] = acc;
  __syncthreads();
  if (slice == 0 && cc < c) {
    float t = 0.f;
#pragma unroll
    for (int s = 0; s < 8; ++s) t += sm[s][cl];
    out[(long long)ni * c + cc] = t / (float)hw;
  }
}

__global__ void k_gap_relu_bwd(const float* __restrict__ dfeat, const float* __restrict__ x, long long hw, int c,
                               long long total, float* __restrict__ dx) {
  long long stride = (long long)gridDim.x * blockDim.x;
  float inv = 1.f / (float)hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int cc = (int)(i % c);
    long long ni = i / ((long long)hw * c);
    dx[i] = x[i] > 0.f ? dfeat[ni * c + cc] * inv : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------------

// ---------------------------------------------------------------------------------------------------
// counter-based random numbers (K21): Philox4x32-10 keyed by `seed`, one 128-bit counter value per group of four outputs;
// uniform in [-1, 1) or standard normal (Box-Muller).  Replaces tf.random.normal of data_utils.py:385 (the latent z) without
// a torch op on the step; the stream position lives in DEVICE memory so that a CUDA-graph replay draws fresh numbers.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t (&o)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}
__global__ void k_philox(float* __restrict__ out, long long n, unsigned long long seed, unsigned long long offset,
                         const unsigned long long* __restrict__ offset_dev, int normal) {
  const unsigned long long base = offset + (offset_dev ? *offset_dev : 0ull);
  const long long groups = (n + 3) / 4, stride = (long long)gridDim.x * blockDim.x;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const unsigned long long ctr = base + (unsigned long long)g;
    uint32_t r[4];
    philox4x32_10((uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    float v[4];
    if (normal) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float u1 = ((float)r[2 * h] + 1.0f) * 2.3283064365386963e-10f;      // (0, 1]
        const float u2 = (float)r[2 * h + 1] * 2.3283064365386963e-10f;           // [0, 1)
        const float rad = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincospif(2.0f * u2, &sn, &cs);
        v[2 * h] = rad * cs;
        v[2 * h + 1] = rad * sn;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = (float)r[j] * 4.656612873077393e-10f - 1.0f;  // [-1, 1)
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * g + j < n) out[4 * g + j] = v[j];
  }
}
__global__ void k_philox_advance(unsigned long long* offset_dev, unsigned long long by) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *offset_dev += by;
}


// ragged batches (several word lengths in one launch): zero everything right of a word's own width
template <typename T>
__global__ void k_mask_width(T* __restrict__ x, long long total4, int h, int w, int c4, const int* __restrict__ lens, int cols_per_char) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += stride) {
    const long long pix = i / c4;
    const int col = (int)(pix % w);
    const int ni = (int)(pix / ((long long)w * h));
    if (col >= lens[ni] * cols_per_char) sg_st4(x + 4 * i, make_float4(0.f, 0.f, 0.f, 0.f));
  }
}
__global__ void k_label_lengths(const int* __restrict__ labels, int b, int l, int* __restrict__ lens) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b) return;
  int n = 0;
  while (n < l && labels[(long long)i * l + n] >= 0) ++n;
  lens[i] = n;
}

extern "C" {

int sg_act_prep(sg_ctx* ctx, const float* x, long long n, void* relu_out, void* copy_out, int out_dt) {
  SG_REQUIRE(ctx && x && n >= 0, "sg_act_prep: bad args");
  if (n == 0) return SG_OK;
  long long n4 = (((uintptr_t)x | (uintptr_t)relu_out | (uintptr_t)copy_out) & 15) == 0 ? n / 4 : 0;
  SG_DISPATCH_DT(out_dt, TO,
                 sg_launch(ctx, k_act_prep<TO>, ew_grid(ctx, n / 4 + 1, 256), 256, 0, x, n4, n, (TO*)relu_out, (TO*)copy_out));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_mask_mul(sg_ctx* ctx, const float* dy, const void* act, int act_dt, void* out, int out_dt, long long n,
                int accumulate) {
  SG_REQUIRE(ctx && dy && act && out && n >= 0, "sg_mask_mul: bad args");
  if (n == 0) return SG_OK;
  long long n4 = (((uintptr_t)dy | (uintptr_t)act | (uintptr_t)out) & 15) == 0 ? n / 4 : 0;
  int grid = ew_grid(ctx, n / 4 + 1, 256);
  SG_DISPATCH_DT(act_dt, TA,
                 SG_DISPATCH_DT(out_dt, TO,
                                sg_launch(ctx, k_mask_mul<TA, TO>, grid, 256, 0, dy, (const TA*)act, (TO*)out, n4, n, accumulate)));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_axpby(sg_ctx* ctx, float a, const float* x, float b, const float* y, float* out, long long n) {
  SG_REQUIRE(ctx && x && out && n >= 0, "sg_axpby: bad args");
  if (n == 0) return SG_OK;
  long long n4 = (((uintptr_t)x | (uintptr_t)y | (uintptr_t)out) & 15) == 0 ? n / 4 : 0;
  sg_launch(ctx, k_axpby, ew_grid(ctx, n / 4 + 1, 256), 256, 0, a, x, b, y, out, n4, n);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_scale_add(sg_ctx* ctx, const float* sigma, const float* a, const float* x, float* out, long long n) {
  SG_REQUIRE(ctx && sigma && a && out && n >= 0, "sg_scale_add: bad args");
  if (n == 0) return SG_OK;
  long long n4 = (((uintptr_t)a | (uintptr_t)x | (uintptr_t)out) & 15) == 0 ? n / 4 : 0;
  sg_launch(ctx, k_scale_add, ew_grid(ctx, n / 4 + 1, 256), 256, 0, sigma, a, x, out, n4, n);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_tanh_fwd(sg_ctx* ctx, const float* x, float* y, long long n) {
  SG_REQUIRE(ctx && x && y && n >= 0, "sg_tanh_fwd: bad args");
  if (n == 0) return SG_OK;
  sg_launch(ctx, k_tanh_fwd, ew_grid(ctx, n, 256), 256, 0, x, y, n);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_tanh_bwd(sg_ctx* ctx, const float* dy, const float* y, float* dx, long long n) {
  SG_REQUIRE(ctx && dy && y && dx && n >= 0, "sg_tanh_bwd: bad args");
  if (n == 0) return SG_OK;
  sg_launch(ctx, k_tanh_bwd, ew_grid(ctx, n, 256), 256, 0, dy, y, dx, n);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_scale_rows(sg_ctx* ctx, float* x, const float* w, int rows, long long cols) {
  SG_REQUIRE(ctx && x && w && rows >= 0 && cols >= 0, "sg_scale_rows: bad args");
  if ((long long)rows * cols == 0) return SG_OK;
  sg_launch(ctx, k_scale_rows, ew_grid(ctx, (long long)rows * cols, 256), 256, 0, x, w, rows, cols);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

/* x[i, :] *= up[i] * mult, i < n; x is [n, per_sample] (fp32 or bf16, per_sample % 8 == 0) */
int sg_scale_samples(sg_ctx* ctx, void* x, int dt, int n, long long per_sample, const float* up, float mult) {
  SG_REQUIRE(ctx && x && up && n >= 0 && per_sample >= 0 && per_sample % 8 == 0 && ((uintptr_t)x & 15) == 0, "sg_scale_samples: bad args");
  if (n == 0 || per_sample == 0) return SG_OK;
  SG_REQUIRE(n <= 65535, "sg_scale_samples: at most 65535 samples");
  long long need = (per_sample / 8 + 255) / 256;
  long long cap = (long long)ctx->num_sms * 8 / n + 1;
  dim3 grid((unsigned)(need < cap ? need : cap), (unsigned)n);
  SG_DISPATCH_DT(dt, T, sg_launch(ctx, k_scale_samples<T>, grid, 256, 0, (T*)x, per_sample / 8, up, mult));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_dot(sg_ctx* ctx, const float* a, const float* b, long long n, float* out, int accumulate) {
  SG_REQUIRE(ctx && a && b && out && n >= 0, "sg_dot: bad args");
  if (n == 0) {
    if (!accumulate) SG_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float), ctx->stream));
    return SG_OK;
  }
  int dot_blocks = ew_grid(ctx, n, 256);
  if (dot_blocks > 1024) dot_blocks = 1024;
  sg_launch(ctx, k_dot, dot_blocks, 256, 0, a, b, n, out, accumulate, ctx->det_scratch, ctx->det_tickets);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_colsum(sg_ctx* ctx, const void* x, int dt, long long rows, int cols, float* out, int accumulate) {
  SG_REQUIRE(ctx && x && out && rows >= 0 && cols > 0, "sg_colsum: bad args");
  if (rows == 0) {
    if (!accumulate) SG_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * cols, ctx->stream));
    return SG_OK;
  }
  SG_REQUIRE(dt == SG_F32 || dt == SG_BF16, "sg_colsum: bad dtype %d", dt);
  if (cols % 4 == 0 && ((uintptr_t)x & 15) == 0) {
    // per-block partial sums are combined in block order by the last block (deterministic; round 1 used float atomics,
    // which also serialised at ~45 ns per same-address add): bound blocks * cols = the floats that block re-reads, and use
    // 1024-thread blocks so that few blocks still keep enough loads in flight
    constexpr int NT = 1024;
    int cgs = cols / 4, cg_per_pass = cgs < NT ? cgs : NT, lanes_r = NT / cg_per_pass;
    long long blocks = (long long)ctx->num_sms * 2;
    long long cap = 65536 / cols;
    if (cap < 8) cap = 8;
    if (blocks > cap) blocks = cap;
    long long min_rpb = 4LL * lanes_r;
    long long rpb = (rows + blocks - 1) / blocks;
    if (rpb < min_rpb) rpb = min_rpb;
    rpb = (rpb + lanes_r - 1) / lanes_r * lanes_r;
    blocks = (rows + rpb - 1) / rpb;
    if (dt == SG_F32)
      sg_launch(ctx, k_colsum_v4<float, NT>, (int)blocks, NT, 0, (const float*)x, rows, cols, rpb, out, accumulate, ctx->det_scratch,
                                                                  ctx->det_tickets);
    else
      sg_launch(ctx, k_colsum_v4<__nv_bfloat16, NT>, (int)blocks, NT, 0, (const __nv_bfloat16*)x, rows, cols, rpb, out, accumulate,
                                                                          ctx->det_scratch, ctx->det_tickets);
    SG_POST_LAUNCH(ctx);
    return SG_OK;
  }
  long long blocks = (long long)ctx->num_sms * 4;
  if (blocks > rows) blocks = rows;
  long long fit = (long long)(SG_DET_SCRATCH_BYTES / sizeof(float)) / cols / 2;
  if (blocks > fit) blocks = fit;
  SG_REQUIRE(blocks >= 1, "sg_colsum: cols=%d too wide", cols);
  long long rpb = (rows + blocks - 1) / blocks;
  blocks = (rows + rpb - 1) / rpb;
  int threads = cols >= 256 ? 256 : (cols >= 128 ? 128 : 64);
  SG_DISPATCH_DT(dt, T, sg_launch(ctx, k_colsum<T>, (int)blocks, threads, 0, (const T*)x, rows, cols, rpb, out, accumulate,
                                                                              ctx->det_scratch, ctx->det_tickets));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_cast(sg_ctx* ctx, const float* x, void* out, int out_dt, long long n) {
  SG_REQUIRE(ctx && x && out && n >= 0, "sg_cast: bad args");
  if (n == 0) return SG_OK;
  SG_DISPATCH_DT(out_dt, TO, sg_launch(ctx, k_cast<TO>, ew_grid(ctx, n, 256), 256, 0, x, (TO*)out, n));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_avgpool2_fwd(sg_ctx* ctx, const float* x, int n, int h, int w, int c, float* out) {
  SG_REQUIRE(ctx && x && out, "sg_avgpool2_fwd: NULL");
  SG_REQUIRE(h % 2 == 0 && w % 2 == 0 && c % 4 == 0, "sg_avgpool2_fwd: needs even h,w and c%%4==0 (h=%d w=%d c=%d)", h, w, c);
  long long total = (long long)n * (h / 2) * (w / 2) * (c / 4);
  if (total == 0) return SG_OK;
  sg_launch(ctx, k_avgpool2_fwd, ew_grid(ctx, total, 256), 256, 0, x, n, h, w, c / 4, out);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_avgpool2_bwd(sg_ctx* ctx, const float* dout, int n, int h, int w, int c, void* dx, int dx_dt) {
  SG_REQUIRE(ctx && dout && dx, "sg_avgpool2_bwd: NULL");
  SG_REQUIRE(h % 2 == 0 && w % 2 == 0 && c % 4 == 0, "sg_avgpool2_bwd: needs even h,w and c%%4==0");
  long long total = (long long)n * h * w * (c / 4);
  if (total == 0) return SG_OK;
  SG_DISPATCH_DT(dx_dt, TO, sg_launch(ctx, k_avgpool2_bwd<TO>, ew_grid(ctx, total / 4, 256), 256, 0, dout, n, h, w, c / 4, (TO*)dx));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_maxpool_fwd(sg_ctx* ctx, const void* x, int dt, int n, int h, int w, int c, int ph, int pw, void* out) {
  SG_REQUIRE(ctx && x && out, "sg_maxpool_fwd: NULL");
  SG_REQUIRE(ph >= 1 && pw >= 1 && h % ph == 0 && w % pw == 0, "sg_maxpool_fwd: h,w must be divisible by the window");
  long long total = (long long)n * (h / ph) * (w / pw) * c;
  if (total == 0) return SG_OK;
  if (c % 4 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)out & 15) == 0) {
    SG_DISPATCH_DT(dt, T, sg_launch(ctx, k_maxpool_fwd_v4<T>, ew_grid(ctx, total / 4, 256), 256, 0, (const T*)x, n, h, w, c / 4, ph, pw, (T*)out));
  } else {
    SG_DISPATCH_DT(dt, T, sg_launch(ctx, k_maxpool_fwd<T>, ew_grid(ctx, total, 256), 256, 0, (const T*)x, n, h, w, c, ph, pw, (T*)out));
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_maxpool_bwd(sg_ctx* ctx, const float* dout, const void* x, int x_dt, int n, int h, int w, int c, int ph,
                   int pw, int relu_mask, void* dx, int dx_dt) {
  SG_REQUIRE(ctx && dout && x && dx, "sg_maxpool_bwd: NULL");
  SG_REQUIRE(ph >= 1 && pw >= 1 && h % ph == 0 && w % pw == 0, "sg_maxpool_bwd: h,w must be divisible by the window");
  long long total = (long long)n * (h / ph) * (w / pw) * c;
  if (total == 0) return SG_OK;
  if (c % 4 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)dx & 15) == 0 && ((uintptr_t)dout & 15) == 0) {
    int grid = ew_grid(ctx, total / 4, 256);
    SG_DISPATCH_DT(x_dt, TX,
                   SG_DISPATCH_DT(dx_dt, TO,
                                  sg_launch(ctx, k_maxpool_bwd_v4<TX, TO>, grid, 256, 0, dout, (const TX*)x, n, h, w, c / 4, ph, pw, relu_mask, (TO*)dx)));
  } else {
    int grid = ew_grid(ctx, total, 256);
    SG_DISPATCH_DT(x_dt, TX,
                   SG_DISPATCH_DT(dx_dt, TO,
                                  sg_launch(ctx, k_maxpool_bwd<TX, TO>, grid, 256, 0, dout, (const TX*)x, n, h, w, c, ph, pw, relu_mask, (TO*)dx)));
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_gap_relu_fwd(sg_ctx* ctx, const float* x, int n, long long hw, int c, float* out) {
  SG_REQUIRE(ctx && x && out && n >= 0 && hw > 0 && c > 0, "sg_gap_relu_fwd: bad args");
  if (n == 0) return SG_OK;
  dim3 grid(sg_div_up(c, 128), n);
  sg_launch(ctx, k_gap_relu_fwd, grid, 1024, 0, x, hw, c, out);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_gap_relu_bwd(sg_ctx* ctx, const float* dfeat, const float* x, int n, long long hw, int c, float* dx) {
  SG_REQUIRE(ctx && dfeat && x && dx && n >= 0 && hw > 0 && c > 0, "sg_gap_relu_bwd: bad args");
  long long total = (long long)n * hw * c;
  if (total == 0) return SG_OK;
  sg_launch(ctx, k_gap_relu_bwd, ew_grid(ctx, total, 256), 256, 0, dfeat, x, hw, c, total, dx);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}


/* out[n] ~ U[-1, 1) (normal = 0) or N(0, 1) (normal = 1) from the Philox stream (seed, offset + *offset_dev); when offset_dev
 * is given it is advanced by ceil(n / 4) afterwards (a second, one-thread launch), so a replayed CUDA graph continues the
 * stream instead of repeating it. */
int sg_random(sg_ctx* ctx, float* out, long long n, unsigned long long seed, unsigned long long offset,
              unsigned long long* offset_dev, int normal) {
  SG_REQUIRE(ctx && out && n >= 0, "sg_random: bad args");
  if (n == 0) return SG_OK;
  long long groups = (n + 3) / 4;
  sg_launch(ctx, k_philox, ew_grid(ctx, groups, 256), 256, 0, out, n, seed, offset, offset_dev, normal);
  SG_POST_LAUNCH(ctx);
  if (offset_dev) {
    sg_launch(ctx, k_philox_advance, 1, 32, 0, offset_dev, (unsigned long long)groups);
    SG_POST_LAUNCH(ctx);
  }
  return SG_OK;
}


/* ragged batches: x[n, :, col, :] = 0 for col >= cols_per_char * lens[n]  (x is NHWC [n,h,w,c], c % 4 == 0) */
int sg_mask_width(sg_ctx* ctx, void* x, int dt, int n, int h, int w, int c, const int* lens, int cols_per_char) {
  SG_REQUIRE(ctx && x && lens && n >= 0 && h > 0 && w > 0 && c > 0 && c % 4 == 0 && cols_per_char > 0, "sg_mask_width: bad args");
  long long total = (long long)n * h * w * (c / 4);
  if (total == 0) return SG_OK;
  SG_DISPATCH_DT(dt, T, sg_launch(ctx, k_mask_width<T>, ew_grid(ctx, total, 256), 256, 0, (T*)x, total, h, w, c / 4, lens, cols_per_char));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

/* lens[b] = number of leading labels >= 0 of row b (padded label matrices of ragged batches use -1) */
int sg_label_lengths(sg_ctx* ctx, const int* labels, int b, int l, int* lens) {
  SG_REQUIRE(ctx && labels && lens && b >= 0 && l > 0, "sg_label_lengths: bad args");
  if (b == 0) return SG_OK;
  sg_launch(ctx, k_label_lengths, sg_div_up(b, 256), 256, 0, labels, b, l, lens);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
