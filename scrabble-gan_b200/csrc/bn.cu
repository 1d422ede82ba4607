// Batch-norm / conditional batch-norm kernels (HBM-bound reductions + apply passes).
// Reference: resnet_ops.py:13-28 (ConditionalBatchNorm), net_architecture.py:42,46,281 (BatchNormalization).
// x is [n, hw, c] fp32 (NHWC flattened), c % 4 == 0, c <= 1024.
#include "common.cuh"

#define BN_MAX_BLOCKS 592

// thread layout shared by the reduction kernels: 256 threads = (256/tc) row lanes x tc channel quads
struct BnLayout {
  int tc, lanes;
};
static inline BnLayout bn_layout(int c) {
  BnLayout l;
  l.tc = c / 4;
  l.lanes = 256 / l.tc;
  if (l.lanes < 1) l.lanes = 1;
  return l;
}

__global__ void k_bn_stats(const float* __restrict__ x, long long rows, int c, int tc, int lanes,
                           long long rows_per_block, float* __restrict__ partial) {
  extern __shared__ float sm[];     // [lanes][2*c]
  int q = threadIdx.x % tc, lane = threadIdx.x / tc;
  long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  float4 s = make_float4(0, 0, 0, 0), ss = make_float4(0, 0, 0, 0);
  if (lane < lanes) {
    for (long long r = r0 + lane; r < r1; r += lanes) {
      float4 v = sg_ld4(x + r * c + 4 * q);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      ss.x += v.x * v.x; ss.y += v.y * v.y; ss.z += v.z * v.z; ss.w += v.w * v.w;
    }
    float* row = sm + (long long)lane * 2 * c;
    sg_st4(row + 4 * q, s);
    sg_st4(row + c + 4 * q, ss);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < 2 * c; j += blockDim.x) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += sm[(long long)l * 2 * c + j];
    partial[(long long)blockIdx.x * 2 * c + j] = t;
  }
}

// second stage of the statistics: block = 32 columns x 16 slices of the per-block partials (double accumulation),
// slices combined through shared memory -- the serial chain per thread is nblocks/16 loads instead of nblocks.
__global__ void __launch_bounds__(512) k_bn_stats_reduce(const float* __restrict__ partial, int nblocks, int c2,
                                                          float* __restrict__ sums) {
  __shared__ double sm[16][33];
  const int jx = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + jx;
  double t = 0.0;
  if (j < c2)
    for (int b = sl; b < nblocks; b += 16) t += (double)partial[(long long)b * c2 + j];
  sm[sl][jx] = t;
  __syncthreads();
  if (sl == 0 && j < c2) {
#pragma unroll
    for (int k = 1; k < 16; ++k) t += sm[k][jx];
    sums[j] = (float)t;
  }
}

__global__ void k_bn_finalize(const float* __restrict__ sums, double count, int c, float eps, float momentum,
                              float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ mm,
                              float* __restrict__ mv) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= c) return;
  double m = (double)sums[j] / count;
  double var = (double)sums[c + j] / count - m * m;
  if (var < 0.0) var = 0.0;
  mean[j] = (float)m;
  rstd[j] = (float)(1.0 / sqrt(var + (double)eps));
  if (mm) mm[j] = mm[j] * momentum + (float)m * (1.f - momentum);
  if (mv) {
    double unb = count > 1.0 ? var * (count / (count - 1.0)) : var;
    mv[j] = mv[j] * momentum + (float)unb * (1.f - momentum);
  }
}

__global__ void k_bn_infer_prepare(const float* __restrict__ mm, const float* __restrict__ mv, int c, float eps,
                                   float* __restrict__ mean, float* __restrict__ rstd) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= c) return;
  mean[j] = mm[j];
  rstd[j] = rsqrtf(mv[j] + eps);
}

template <typename TO>
__global__ void k_bn_apply(const float* __restrict__ x, long long total4, long long hw, int c4,
                           const float* __restrict__ mean, const float* __restrict__ rstd,
                           const float* __restrict__ gamma, const float* __restrict__ beta, long long gb_stride,
                           int relu, TO* __restrict__ out) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += stride) {
    int q = (int)(i % c4);
    long long ni = i / (hw * c4);
    float4 v = sg_ld4(x + 4 * i), m = sg_ld4(mean + 4 * q), r = sg_ld4(rstd + 4 * q);
    float4 g = gamma ? sg_ld4(gamma + ni * gb_stride + 4 * q) : make_float4(1, 1, 1, 1);
    float4 b = beta ? sg_ld4(beta + ni * gb_stride + 4 * q) : make_float4(0, 0, 0, 0);
    float4 y = make_float4((v.x - m.x) * r.x * g.x + b.x, (v.y - m.y) * r.y * g.y + b.y,
                           (v.z - m.z) * r.z * g.z + b.z, (v.w - m.w) * r.w * g.w + b.w);
    if (relu) y = make_float4(fmaxf(y.x, 0.f), fmaxf(y.y, 0.f), fmaxf(y.z, 0.f), fmaxf(y.w, 0.f));
    sg_st4(out + 4 * i, y);
  }
}

template <typename TA>
__global__ void k_bn_bwd_reduce(const float* __restrict__ dy, const TA* __restrict__ act, const float* __restrict__ x,
                                long long hw, int c, int tc, int lanes, long long rows_per_block,
                                const float* __restrict__ mean, const float* __restrict__ rstd,
                                float* __restrict__ s1, float* __restrict__ s2, float* __restrict__ scratch,
                                unsigned int* __restrict__ tickets) {
  extern __shared__ float sm[];     // [lanes][2*c]
  int ni = blockIdx.y;
  int q = threadIdx.x % tc, lane = threadIdx.x / tc;
  long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = r0 + rows_per_block;
  if (r1 > hw) r1 = hw;
  float4 a = make_float4(0, 0, 0, 0), b = make_float4(0, 0, 0, 0);
  if (lane < lanes) {
    float4 m = sg_ld4(mean + 4 * q), r = sg_ld4(rstd + 4 * q);
    for (long long p = r0 + lane; p < r1; p += lanes) {
      long long off = ((long long)ni * hw + p) * c + 4 * q;
      float4 d = sg_ld4(dy + off);
      if (act) {
        float4 t = sg_ld4(act + off);
        d.x = t.x > 0.f ? d.x : 0.f; d.y = t.y > 0.f ? d.y : 0.f; d.z = t.z > 0.f ? d.z : 0.f; d.w = t.w > 0.f ? d.w : 0.f;
      }
      float4 v = sg_ld4(x + off);
      a.x += d.x; a.y += d.y; a.z += d.z; a.w += d.w;
      b.x += d.x * (v.x - m.x) * r.x; b.y += d.y * (v.y - m.y) * r.y;
      b.z += d.z * (v.z - m.z) * r.z; b.w += d.w * (v.w - m.w) * r.w;
    }
    float* row = sm + (long long)lane * 2 * c;
    sg_st4(row + 4 * q, a);
    sg_st4(row + c + 4 * q, b);
  }
  __syncthreads();
  // deterministic combine over the gridDim.x row slabs of sample ni (common.cuh, scheme B); s1 / s2 are overwritten
  float* slots = scratch + (long long)ni * gridDim.x * 2 * c;
  for (int j = threadIdx.x; j < 2 * c; j += blockDim.x) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += sm[(long long)l * 2 * c + j];
    if (gridDim.x == 1) {
      if (j < c) s1[(long long)ni * c + j] = t;
      else s2[(long long)ni * c + (j - c)] = t;
    } else {
      slots[(long long)blockIdx.x * 2 * c + j] = t;
    }
  }
  if (gridDim.x == 1) return;
  if (!sg_det_arrive_last(tickets + ni, gridDim.x)) return;      // gridDim.x <= 32: one level
  sg_det_block_reduce(slots, gridDim.x, 2 * c, [&](int j, float t) {
    if (j < c) s1[(long long)ni * c + j] = t;
    else s2[(long long)ni * c + (j - c)] = t;
  });
}

// block = 32 channels x 8 sample slices, slices combined through shared memory
__global__ void __launch_bounds__(256) k_bn_bwd_combine(const float* __restrict__ s1, const float* __restrict__ s2,
                                                         const float* __restrict__ gamma, long long gb_stride, int n, int c,
                                                         float* __restrict__ ab) {
  __shared__ float sa[8][33], sb[8][33];
  const int jx = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + jx;
  float a = 0.f, b = 0.f;
  if (j < c)
    for (int i = sl; i < n; i += 8) {
      float g = gamma ? gamma[(long long)i * gb_stride + j] : 1.f;
      a += g * s1[(long long)i * c + j];
      b += g * s2[(long long)i * c + j];
    }
  sa[sl][jx] = a;
  sb[sl][jx] = b;
  __syncthreads();
  if (sl == 0 && j < c) {
#pragma unroll
    for (int k = 1; k < 8; ++k) { a += sa[k][jx]; b += sb[k][jx]; }
    ab[j] = a;
    ab[c + j] = b;
  }
}

template <typename TA, typename TO>
__global__ void k_bn_bwd_apply(const float* __restrict__ dy, const TA* __restrict__ act, const float* __restrict__ x,
                               long long total4, long long hw, int c4, const float* __restrict__ mean,
                               const float* __restrict__ rstd, const float* __restrict__ gamma, long long gb_stride,
                               const float* __restrict__ ab, float inv_count, int use_batch, int mask_by_x,
                               TO* __restrict__ dx, int accumulate) {
  long long stride = (long long)gridDim.x * blockDim.x;
  int c = 4 * c4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += stride) {
    int q = (int)(i % c4);
    long long ni = i / (hw * c4);
    float4 d = sg_ld4(dy + 4 * i);
    if (act) {
      float4 t = sg_ld4(act + 4 * i);
      d.x = t.x > 0.f ? d.x : 0.f; d.y = t.y > 0.f ? d.y : 0.f; d.z = t.z > 0.f ? d.z : 0.f; d.w = t.w > 0.f ? d.w : 0.f;
    }
    float4 r = sg_ld4(rstd + 4 * q);
    float4 g = gamma ? sg_ld4(gamma + ni * gb_stride + 4 * q) : make_float4(1, 1, 1, 1);
    float4 o = make_float4(g.x * d.x, g.y * d.y, g.z * d.z, g.w * d.w);
    float4 v = make_float4(1, 1, 1, 1);
    if (use_batch || mask_by_x) v = sg_ld4(x + 4 * i);
    if (use_batch) {
      float4 m = sg_ld4(mean + 4 * q);
      float4 a0 = sg_ld4(ab + 4 * q), a1 = sg_ld4(ab + c + 4 * q);
      o.x -= (a0.x + (v.x - m.x) * r.x * a1.x) * inv_count;
      o.y -= (a0.y + (v.y - m.y) * r.y * a1.y) * inv_count;
      o.z -= (a0.z + (v.z - m.z) * r.z * a1.z) * inv_count;
      o.w -= (a0.w + (v.w - m.w) * r.w * a1.w) * inv_count;
    }
    o.x *= r.x; o.y *= r.y; o.z *= r.z; o.w *= r.w;
    if (mask_by_x) {
      o.x = v.x > 0.f ? o.x : 0.f; o.y = v.y > 0.f ? o.y : 0.f; o.z = v.z > 0.f ? o.z : 0.f; o.w = v.w > 0.f ? o.w : 0.f;
    }
    if (accumulate) {
      float4 p = sg_ld4(dx + 4 * i);
      o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
    }
    sg_st4(dx + 4 * i, o);
  }
}

static inline int bn_grid(sg_ctx* ctx, long long items) {
  long long need = (items + 255) / 256, cap = (long long)ctx->num_sms * 8;
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}

extern "C" {

size_t sg_bn_stats_scratch_bytes(long long rows, int c) {
  (void)rows;
  return (size_t)BN_MAX_BLOCKS * 2 * (size_t)c * sizeof(float);
}

int sg_bn_stats(sg_ctx* ctx, const float* x, long long rows, int c, float* sums, void* scratch, size_t scratch_bytes) {
  SG_REQUIRE(ctx && x && sums && scratch, "sg_bn_stats: NULL");
  SG_REQUIRE(c % 4 == 0 && c >= 4 && c <= 1024, "sg_bn_stats: c=%d must be a multiple of 4 in [4,1024]", c);
  SG_REQUIRE(scratch_bytes >= sg_bn_stats_scratch_bytes(rows, c), "sg_bn_stats: scratch too small");
  SG_REQUIRE(rows > 0, "sg_bn_stats: rows must be > 0");
  BnLayout l = bn_layout(c);
  long long blocks = (long long)ctx->num_sms * 4;
  if (blocks > BN_MAX_BLOCKS) blocks = BN_MAX_BLOCKS;
  long long min_rows = 4LL * l.lanes;
  if (blocks > (rows + min_rows - 1) / min_rows) blocks = (rows + min_rows - 1) / min_rows;
  long long rpb = (rows + blocks - 1) / blocks;
  blocks = (rows + rpb - 1) / rpb;
  size_t smem = (size_t)l.lanes * 2 * c * sizeof(float);
  sg_launch(ctx, k_bn_stats, (int)blocks, 256, smem, x, rows, c, l.tc, l.lanes, rpb, (float*)scratch);
  SG_POST_LAUNCH(ctx);
  sg_launch(ctx, k_bn_stats_reduce, sg_div_up(2 * c, 32), 512, 0, (const float*)scratch, (int)blocks, 2 * c, sums);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

/* stage 1 only (per-block partial sums into scratch, at most one block per SM): the second stage, the cross-replica
 * exchange and the finalisation are fused in sg_bn_finalize_peer (peer.cu) */
int sg_bn_stats_partial(sg_ctx* ctx, const float* x, long long rows, int c, void* scratch, size_t scratch_bytes, int* nblocks_out) {
  SG_REQUIRE(ctx && x && scratch && nblocks_out, "sg_bn_stats_partial: NULL");
  SG_REQUIRE(c % 4 == 0 && c >= 4 && c <= 1024, "sg_bn_stats_partial: c=%d must be a multiple of 4 in [4,1024]", c);
  SG_REQUIRE(rows > 0, "sg_bn_stats_partial: rows must be > 0");
  BnLayout l = bn_layout(c);
  long long blocks = ctx->num_sms;
  long long min_rows = 4LL * l.lanes;
  if (blocks > (rows + min_rows - 1) / min_rows) blocks = (rows + min_rows - 1) / min_rows;
  long long rpb = (rows + blocks - 1) / blocks;
  blocks = (rows + rpb - 1) / rpb;
  SG_REQUIRE(scratch_bytes >= (size_t)blocks * 2 * c * sizeof(float), "sg_bn_stats_partial: scratch too small");
  size_t smem = (size_t)l.lanes * 2 * c * sizeof(float);
  sg_launch(ctx, k_bn_stats, (int)blocks, 256, smem, x, rows, c, l.tc, l.lanes, rpb, (float*)scratch);
  SG_POST_LAUNCH(ctx);
  *nblocks_out = (int)blocks;
  return SG_OK;
}

int sg_bn_finalize(sg_ctx* ctx, const float* sums, double count, int c, float eps, float momentum, float* mean,
                   float* rstd, float* moving_mean, float* moving_var) {
  SG_REQUIRE(ctx && sums && mean && rstd && count > 0 && c > 0, "sg_bn_finalize: bad args");
  sg_launch(ctx, k_bn_finalize, sg_div_up(c, 128), 128, 0, sums, count, c, eps, momentum, mean, rstd, moving_mean, moving_var);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_bn_infer_prepare(sg_ctx* ctx, const float* moving_mean, const float* moving_var, int c, float eps, float* mean,
                        float* rstd) {
  SG_REQUIRE(ctx && moving_mean && moving_var && mean && rstd && c > 0, "sg_bn_infer_prepare: bad args");
  sg_launch(ctx, k_bn_infer_prepare, sg_div_up(c, 128), 128, 0, moving_mean, moving_var, c, eps, mean, rstd);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_bn_apply(sg_ctx* ctx, const float* x, int n, long long hw, int c, const float* mean, const float* rstd,
                const float* gamma, const float* beta, long long gb_stride, int relu, void* out, int out_dt) {
  SG_REQUIRE(ctx && x && mean && rstd && out, "sg_bn_apply: NULL");
  SG_REQUIRE(c % 4 == 0 && (gb_stride == 0 || gb_stride % 4 == 0), "sg_bn_apply: c and gb_stride must be multiples of 4");
  long long total4 = (long long)n * hw * (c / 4);
  if (total4 == 0) return SG_OK;
  SG_DISPATCH_DT(out_dt, TO,
                 sg_launch(ctx, k_bn_apply<TO>, bn_grid(ctx, total4), 256, 0, x, total4, hw, c / 4, mean, rstd, gamma, beta,
                                                                               gb_stride, relu, (TO*)out));
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_bn_bwd_reduce(sg_ctx* ctx, const float* dy, const void* act, int act_dt, const float* x, int n, long long hw,
                     int c, const float* mean, const float* rstd, float* s1, float* s2) {
  SG_REQUIRE(ctx && dy && x && mean && rstd && s1 && s2, "sg_bn_bwd_reduce: NULL");
  SG_REQUIRE(c % 4 == 0 && c >= 4 && c <= 1024, "sg_bn_bwd_reduce: c=%d must be a multiple of 4 in [4,1024]", c);
  if ((long long)n * hw == 0) {
    SG_CHECK_CUDA(cudaMemsetAsync(s1, 0, sizeof(float) * (size_t)n * c, ctx->stream));
    SG_CHECK_CUDA(cudaMemsetAsync(s2, 0, sizeof(float) * (size_t)n * c, ctx->stream));
    return SG_OK;
  }
  SG_REQUIRE(n <= SG_DET_TICKETS, "sg_bn_bwd_reduce: batch %d too large", n);
  BnLayout l = bn_layout(c);
  long long blocks = ((long long)ctx->num_sms * 4 + n - 1) / n;
  long long min_rows = 4LL * l.lanes;
  if (blocks > (hw + min_rows - 1) / min_rows) blocks = (hw + min_rows - 1) / min_rows;
  long long fit = (long long)(SG_DET_SCRATCH_BYTES / sizeof(float)) / ((long long)n * 2 * c);      // per-block partial slots
  if (blocks > fit) blocks = fit;
  if (blocks > 32) blocks = 32;
  if (blocks < 1) blocks = 1;
  long long rpb = (hw + blocks - 1) / blocks;
  blocks = (hw + rpb - 1) / rpb;
  size_t smem = (size_t)l.lanes * 2 * c * sizeof(float);
  dim3 grid((unsigned)blocks, (unsigned)n);
  if (act) {
    SG_DISPATCH_DT(act_dt, TA,
                   sg_launch(ctx, k_bn_bwd_reduce<TA>, grid, 256, smem, dy, (const TA*)act, x, hw, c, l.tc, l.lanes, rpb, mean, rstd, s1, s2,
                                                                         ctx->det_scratch, ctx->det_tickets));
  } else {
    sg_launch(ctx, k_bn_bwd_reduce<float>, grid, 256, smem, dy, nullptr, x, hw, c, l.tc, l.lanes, rpb, mean, rstd, s1, s2, ctx->det_scratch,
                                                             ctx->det_tickets);
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_bn_bwd_combine(sg_ctx* ctx, const float* s1, const float* s2, const float* gamma, long long gb_stride, int n,
                      int c, float* ab) {
  SG_REQUIRE(ctx && s1 && s2 && ab && c > 0, "sg_bn_bwd_combine: bad args");
  sg_launch(ctx, k_bn_bwd_combine, sg_div_up(c, 32), 256, 0, s1, s2, gamma, gb_stride, n, c, ab);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_bn_bwd_apply(sg_ctx* ctx, const float* dy, const void* act, int act_dt, const float* x, int n, long long hw,
                    int c, const float* mean, const float* rstd, const float* gamma, long long gb_stride,
                    const float* ab, double count, int use_batch_terms, int mask_by_x, void* dx, int dx_dt,
                    int accumulate) {
  SG_REQUIRE(ctx && dy && x && mean && rstd && dx, "sg_bn_bwd_apply: NULL");
  SG_REQUIRE(!use_batch_terms || (ab && count > 0), "sg_bn_bwd_apply: batch terms need ab and count");
  SG_REQUIRE(c % 4 == 0 && (gb_stride == 0 || gb_stride % 4 == 0), "sg_bn_bwd_apply: c and gb_stride must be multiples of 4");
  SG_REQUIRE(!accumulate || dx_dt == SG_F32, "sg_bn_bwd_apply: accumulate needs fp32 dx");
  long long total4 = (long long)n * hw * (c / 4);
  if (total4 == 0) return SG_OK;
  float inv = use_batch_terms ? (float)(1.0 / count) : 0.f;
  int grid = bn_grid(ctx, total4);
  if (act) {
    SG_DISPATCH_DT(act_dt, TA,
                   SG_DISPATCH_DT(dx_dt, TO,
                                  sg_launch(ctx, k_bn_bwd_apply<TA, TO>, grid, 256, 0, dy, (const TA*)act, x, total4, hw, c / 4, mean, rstd, gamma,
                                                                                        gb_stride, ab, inv, use_batch_terms, mask_by_x, (TO*)dx, accumulate)));
  } else {
    SG_DISPATCH_DT(dx_dt, TO,
                   sg_launch(ctx, k_bn_bwd_apply<float, TO>, grid, 256, 0, dy, nullptr, x, total4, hw, c / 4, mean, rstd, gamma, gb_stride,
                                                                            ab, inv, use_batch_terms, mask_by_x, (TO*)dx, accumulate));
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
