// Fused optimizer updates over flat parameter buffers (K19) and spectral norm (K18).
// Reference: main.py:25-35 (tf.keras.optimizers.Adam(lr, beta_1, beta_2) x4, optional RMSprop for R),
// data_utils.py:451-468 (apply_gradients), arch_ops.py:99-126 (spectral_norm).
// Keras Adam:    m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  w -= lr_t m / (sqrt(v) + eps),
//                lr_t = lr sqrt(1-b2^t)/(1-b1^t) (computed on the host), eps = 1e-7 OUTSIDE the sqrt.
// Keras RMSprop: ms = rho ms + (1-rho) g^2;  w -= lr g / (sqrt(ms) + eps).
// HBM-bound: 4 reads + 3 writes per parameter, float4-vectorised.
#include "common.cuh"

// wb (optional): bf16 mirror of w, written in the same pass -- the tensor-core convs read their filters from it in place
__global__ void k_adam(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                       long long n4, long long n, float lr_t, float b1, float b2, float eps, __nv_bfloat16* __restrict__ wb,
                       const float* __restrict__ lr_dev) {
  if (lr_dev) lr_t = *lr_dev;          // step size from device memory (CUDA-graph replays: see k_adam_prepare)
  long long stride = (long long)gridDim.x * blockDim.x;
  const float c1 = 1.f - b1, c2 = 1.f - b2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 gw = sg_ld4(g + 4 * i), mw = sg_ld4(m + 4 * i), vw = sg_ld4(v + 4 * i), ww = sg_ld4(w + 4 * i);
    mw.x = b1 * mw.x + c1 * gw.x; mw.y = b1 * mw.y + c1 * gw.y; mw.z = b1 * mw.z + c1 * gw.z; mw.w = b1 * mw.w + c1 * gw.w;
    vw.x = b2 * vw.x + c2 * gw.x * gw.x; vw.y = b2 * vw.y + c2 * gw.y * gw.y;
    vw.z = b2 * vw.z + c2 * gw.z * gw.z; vw.w = b2 * vw.w + c2 * gw.w * gw.w;
    ww.x -= lr_t * mw.x / (sqrtf(vw.x) + eps); ww.y -= lr_t * mw.y / (sqrtf(vw.y) + eps);
    ww.z -= lr_t * mw.z / (sqrtf(vw.z) + eps); ww.w -= lr_t * mw.w / (sqrtf(vw.w) + eps);
    sg_st4(m + 4 * i, mw); sg_st4(v + 4 * i, vw); sg_st4(w + 4 * i, ww);
    if (wb) sg_st4(wb + 4 * i, ww);
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float gi = g[i];
    float mi = b1 * m[i] + c1 * gi, vi = b2 * v[i] + c2 * gi * gi;
    m[i] = mi; v[i] = vi;
    float wi = w[i] - lr_t * mi / (sqrtf(vi) + eps);
    w[i] = wi;
    if (wb) wb[i] = __float2bfloat16_rn(wi);
  }
}

// The step's own optimizer launch (train_step's fused apply_gradients): as k_adam, plus
//   * beta1 == 0 (the reference's configuration, scrabble_gan.gin:8: m_t = g_t exactly): the first-moment slot is neither read
//     nor written -- no later step can observe it -- which removes 8 of the 30 bytes per parameter;
//   * clear_g: the consumed gradient is overwritten with zeros in the same pass, so the next step needs no memset of the bucket.
template <bool kNoM, bool kClear>
__global__ void k_adam_fused(float* __restrict__ w, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n4,
                             long long n, float b1, float b2, float eps, __nv_bfloat16* __restrict__ wb, const float* __restrict__ lr_dev) {
  const float lr_t = *lr_dev;
  long long stride = (long long)gridDim.x * blockDim.x;
  const float c1 = 1.f - b1, c2 = 1.f - b2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 gw = sg_ld4(g + 4 * i), vw = sg_ld4(v + 4 * i), ww = sg_ld4(w + 4 * i), mw = gw;
    if (!kNoM) {
      mw = sg_ld4(m + 4 * i);
      mw.x = b1 * mw.x + c1 * gw.x; mw.y = b1 * mw.y + c1 * gw.y; mw.z = b1 * mw.z + c1 * gw.z; mw.w = b1 * mw.w + c1 * gw.w;
      sg_st4(m + 4 * i, mw);
    }
    vw.x = b2 * vw.x + c2 * gw.x * gw.x; vw.y = b2 * vw.y + c2 * gw.y * gw.y;
    vw.z = b2 * vw.z + c2 * gw.z * gw.z; vw.w = b2 * vw.w + c2 * gw.w * gw.w;
    ww.x -= lr_t * mw.x / (sqrtf(vw.x) + eps); ww.y -= lr_t * mw.y / (sqrtf(vw.y) + eps);
    ww.z -= lr_t * mw.z / (sqrtf(vw.z) + eps); ww.w -= lr_t * mw.w / (sqrtf(vw.w) + eps);
    sg_st4(v + 4 * i, vw); sg_st4(w + 4 * i, ww);
    if (wb) sg_st4(wb + 4 * i, ww);
    if (kClear) sg_st4(g + 4 * i, make_float4(0.f, 0.f, 0.f, 0.f));
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float gi = g[i], mi = gi;
    if (!kNoM) { mi = b1 * m[i] + c1 * gi; m[i] = mi; }
    float vi = b2 * v[i] + c2 * gi * gi;
    v[i] = vi;
    float wi = w[i] - lr_t * mi / (sqrtf(vi) + eps);
    w[i] = wi;
    if (wb) wb[i] = __float2bfloat16_rn(wi);
    if (kClear) g[i] = 0.f;
  }
}

// Device-side step counter and Keras step size  lr_t = lr sqrt(1 - b2^t) / (1 - b1^t):  t_set >= 0 sets the counter (eager
// calls pass the host iteration count), t_set < 0 increments it (captured launches: every graph replay advances by one).
__global__ void k_adam_prepare(int* __restrict__ step, float* __restrict__ lr_dev, int t_set, float lr, float b1, float b2) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int t = t_set >= 0 ? t_set : *step + 1;
    *step = t;
    double c1 = 1.0 - pow((double)b1, (double)t), c2 = 1.0 - pow((double)b2, (double)t);
    *lr_dev = (float)((double)lr * sqrt(c2) / c1);
  }
}

__global__ void k_rmsprop(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ ms, long long n,
                          float lr, float rho, float eps) {
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float gi = g[i];
    float s = rho * ms[i] + (1.f - rho) * gi * gi;
    ms[i] = s;
    w[i] -= lr * gi / (sqrtf(s) + eps);
  }
}

// ---- spectral norm ----------------------------------------------------------------------------------
// v_raw[r] = sum_c u[c] W[r,c]  (one warp per row)
__global__ void k_sn_rowdot(const float* __restrict__ w, int rows, int cols, const float* __restrict__ u,
                            const float* __restrict__ u_scale, float* __restrict__ v) {
  int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  int lane = threadIdx.x & 31;
  float acc = 0.f;
  for (int c = lane; c < cols; c += 32) acc += u[c] * w[(long long)r * cols + c];
  acc = sg_warp_sum(acc);
  if (lane == 0) v[r] = acc * (u_scale ? *u_scale : 1.f);
}
// t[c] = sum_r v[r] * v_scale * W[r,c]: row slabs (blockIdx.y) are combined in slab order by the last block of each column
// block to arrive (common.cuh, scheme B: deterministic)
__global__ void k_sn_coldot(const float* __restrict__ w, int rows, int cols, const float* __restrict__ v,
                            const float* __restrict__ v_scale, int rows_per_block, float* __restrict__ t,
                            float* __restrict__ scratch, unsigned int* __restrict__ tickets) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  int r0 = blockIdx.y * rows_per_block, r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  float acc = 0.f;
  if (c < cols)
    for (int r = r0; r < r1; ++r) acc += v[r] * w[(long long)r * cols + c];
  float* slots = scratch + (long long)blockIdx.x * gridDim.y * blockDim.x;
  slots[(long long)blockIdx.y * blockDim.x + threadIdx.x] = acc * (*v_scale);
  if (!sg_det_arrive_last(tickets + blockIdx.x, gridDim.y)) return;      // gridDim.y <= 32: one level
  sg_det_block_reduce(slots, gridDim.y, blockDim.x, [&](int j, float sum) {
    int cc = blockIdx.x * blockDim.x + j;
    if (cc < cols) t[cc] = sum;
  });
}
// out[0] = rsqrt(max(sum x^2, 1e-12))   (tf.nn.l2_normalize scale), out[1] = sum x^2
__global__ void k_sn_invnorm(const float* __restrict__ x, int n, float* __restrict__ out) {
  __shared__ float sm[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += x[i] * x[i];
  float t = sg_block_sum(acc, sm);
  if (threadIdx.x == 0) { out[0] = rsqrtf(fmaxf(t, 1e-12f)); out[1] = t; }
}
// sigma = (v W) . u_hat = sum_c t[c] * (t[c]*inv_t) ; u_out = t*inv_t
__global__ void k_sn_sigma(const float* __restrict__ t, int cols, const float* __restrict__ inv_t, float* __restrict__ u_out,
                           float* __restrict__ sigma) {
  __shared__ float sm[32];
  float s = *inv_t, acc = 0.f;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) {
    float uh = t[i] * s;
    if (u_out) u_out[i] = uh;
    acc += t[i] * uh;
  }
  float r = sg_block_sum(acc, sm);
  if (threadIdx.x == 0) *sigma = r;
}
__global__ void k_sn_scale(const float* __restrict__ w, long long n, const float* __restrict__ sigma, float* __restrict__ out) {
  float inv = 1.f / *sigma;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = w[i] * inv;
}

extern "C" {

static int adam_impl(sg_ctx* ctx, float* w, const float* g, float* m, float* v, void* wb, long long n, float lr_t, float beta1,
                     float beta2, float eps, const float* lr_dev = nullptr) {
  SG_REQUIRE(ctx && w && g && m && v && n >= 0, "sg_adam: bad args");
  if (n == 0) return SG_OK;
  long long n4 = (((uintptr_t)w | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v | (uintptr_t)wb) & 15) == 0 ? n / 4 : 0;
  long long need = (n / 4 + 256) / 256, cap = (long long)ctx->num_sms * 8;
  sg_launch(ctx, k_adam, (int)(need < cap ? need : cap), 256, 0, w, g, m, v, n4, n, lr_t, beta1, beta2, eps, (__nv_bfloat16*)wb, lr_dev);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_adam(sg_ctx* ctx, float* w, const float* g, float* m, float* v, long long n, float lr_t, float beta1, float beta2,
            float eps) {
  return adam_impl(ctx, w, g, m, v, nullptr, n, lr_t, beta1, beta2, eps);
}

/* Adam that also refreshes the bf16 mirror of the weights in the same pass (see sg_conv_fwd_tc_direct) */
int sg_adam_mirror(sg_ctx* ctx, float* w, const float* g, float* m, float* v, void* w_mirror_bf16, long long n, float lr_t,
                   float beta1, float beta2, float eps) {
  SG_REQUIRE(w_mirror_bf16 != nullptr, "sg_adam_mirror: NULL mirror");
  return adam_impl(ctx, w, g, m, v, w_mirror_bf16, n, lr_t, beta1, beta2, eps);
}

/* step size kept on the device so that the update can be replayed from a CUDA graph: sg_adam_prepare sets (t >= 0) or
 * advances (t < 0) the device step counter and writes lr_t; sg_adam_dev is sg_adam[_mirror] reading lr_t from lr_dev */
int sg_adam_prepare(sg_ctx* ctx, int* step_dev, float* lr_dev, int t, float lr, float beta1, float beta2) {
  SG_REQUIRE(ctx && step_dev && lr_dev, "sg_adam_prepare: NULL");
  sg_launch(ctx, k_adam_prepare, 1, 32, 0, step_dev, lr_dev, t, lr, beta1, beta2);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_adam_dev(sg_ctx* ctx, float* w, const float* g, float* m, float* v, void* w_mirror_bf16, long long n, const float* lr_dev,
                float beta1, float beta2, float eps) {
  SG_REQUIRE(lr_dev != nullptr, "sg_adam_dev: NULL lr_dev");
  return adam_impl(ctx, w, g, m, v, w_mirror_bf16, n, 0.f, beta1, beta2, eps, lr_dev);
}

/* the train step's optimizer launch: sg_adam_dev that (i) skips the first-moment slot when beta1 == 0 (m_t = g_t: the slot is then
 * not maintained) and (ii) with clear_grad overwrites the consumed gradient with zeros (the next step needs no memset) */
int sg_adam_fused(sg_ctx* ctx, float* w, float* g, float* m, float* v, void* w_mirror_bf16, long long n, const float* lr_dev,
                  float beta1, float beta2, float eps, int clear_grad) {
  SG_REQUIRE(ctx && w && g && m && v && lr_dev && n >= 0, "sg_adam_fused: bad args");
  if (n == 0) return SG_OK;
  long long n4 = (((uintptr_t)w | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v | (uintptr_t)w_mirror_bf16) & 15) == 0 ? n / 4 : 0;
  long long need = (n / 4 + 256) / 256, cap = (long long)ctx->num_sms * 8;
  int grid = (int)(need < cap ? need : cap);
  __nv_bfloat16* wb = (__nv_bfloat16*)w_mirror_bf16;
  if (beta1 == 0.f) {
    if (clear_grad) sg_launch(ctx, k_adam_fused<true, true>, grid, 256, 0, w, g, m, v, n4, n, beta1, beta2, eps, wb, lr_dev);
    else sg_launch(ctx, k_adam_fused<true, false>, grid, 256, 0, w, g, m, v, n4, n, beta1, beta2, eps, wb, lr_dev);
  } else {
    if (clear_grad) sg_launch(ctx, k_adam_fused<false, true>, grid, 256, 0, w, g, m, v, n4, n, beta1, beta2, eps, wb, lr_dev);
    else sg_launch(ctx, k_adam_fused<false, false>, grid, 256, 0, w, g, m, v, n4, n, beta1, beta2, eps, wb, lr_dev);
  }
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_rmsprop(sg_ctx* ctx, float* w, const float* g, float* ms, long long n, float lr, float rho, float eps) {
  SG_REQUIRE(ctx && w && g && ms && n >= 0, "sg_rmsprop: bad args");
  if (n == 0) return SG_OK;
  long long need = (n + 255) / 256, cap = (long long)ctx->num_sms * 8;
  sg_launch(ctx, k_rmsprop, (int)(need < cap ? need : cap), 256, 0, w, g, ms, n, lr, rho, eps);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_spectral_norm(sg_ctx* ctx, const float* w, int rows, int cols, const float* u, int power_iteration, float* w_out,
                     float* u_out, float* sigma_out, float* scratch) {
  SG_REQUIRE(ctx && w && u && w_out && sigma_out && scratch, "sg_spectral_norm: NULL");
  SG_REQUIRE(rows > 0 && cols > 0 && power_iteration >= 1, "sg_spectral_norm: bad sizes");
  float* v = scratch;                 // [rows]
  float* t = scratch + rows;          // [cols]
  float* sc = scratch + rows + cols;  // [4]: inv_v, |v|^2, inv_t, |t|^2
  const float* u_cur = u;
  const float* u_scale = nullptr;
  for (int it = 0; it < power_iteration; ++it) {
    sg_launch(ctx, k_sn_rowdot, sg_div_up(rows, 8), 256, 0, w, rows, cols, u_cur, u_scale, v);
    SG_POST_LAUNCH(ctx);
    sg_launch(ctx, k_sn_invnorm, 1, 1024, 0, v, rows, sc);
    SG_POST_LAUNCH(ctx);
    int slabs = sg_div_up(rows, 64);
    if (slabs > 32) slabs = 32;
    SG_REQUIRE(sg_div_up(cols, 128) <= SG_DET_TICKETS, "sg_spectral_norm: too many columns");
    {
      long long fit = (long long)(SG_DET_SCRATCH_BYTES / sizeof(float)) / ((long long)sg_div_up(cols, 128) * 128);
      if (slabs > fit) slabs = (int)fit;
      if (slabs < 1) slabs = 1;
    }
    int rpb = sg_div_up(rows, slabs);
    slabs = sg_div_up(rows, rpb);
    dim3 grid(sg_div_up(cols, 128), slabs);
    sg_launch(ctx, k_sn_coldot, grid, 128, 0, w, rows, cols, v, sc, rpb, t, ctx->det_scratch, ctx->det_tickets);
    SG_POST_LAUNCH(ctx);
    sg_launch(ctx, k_sn_invnorm, 1, 1024, 0, t, cols, sc + 2);
    SG_POST_LAUNCH(ctx);
    u_cur = t;            // next iteration uses u_hat = t * inv_t
    u_scale = sc + 2;
    if (it + 1 < power_iteration) {
      // materialise u_hat so that t can be reused
      SG_REQUIRE(u_out != nullptr, "sg_spectral_norm: power_iteration > 1 needs u_out as a staging buffer");
      sg_launch(ctx, k_sn_sigma, 1, 1024, 0, t, cols, sc + 2, u_out, sigma_out);
      SG_POST_LAUNCH(ctx);
      u_cur = u_out;
      u_scale = nullptr;
    }
  }
  sg_launch(ctx, k_sn_sigma, 1, 1024, 0, t, cols, sc + 2, u_out, sigma_out);
  SG_POST_LAUNCH(ctx);
  long long n = (long long)rows * cols;
  long long need = (n + 255) / 256, cap = (long long)ctx->num_sms * 8;
  sg_launch(ctx, k_sn_scale, (int)(need < cap ? need : cap), 256, 0, w, n, sigma_out, w_out);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// Spectral-norm weight re-parameterisation, backward (paper-faithful option `apply_sn`, SURVEY Q2 / section 8f):
//     W_sn = W / sigma,  sigma = v^T W u  with the power-iteration vectors u, v treated as constants
//     dL/dW = ( G - <G, W_sn> v u^T ) / sigma,   G = dL/dW_sn   (in place on g)
// v_raw / inv_v are what sg_spectral_norm leaves in its scratch (v_hat = v_raw * inv_v), u_hat its u_out.
// ---------------------------------------------------------------------------------------------------
__global__ void k_sn_bwd(float* __restrict__ g, const float* __restrict__ dot, const float* __restrict__ v_raw,
                         const float* __restrict__ inv_v, const float* __restrict__ u_hat, const float* __restrict__ sigma, int rows,
                         int cols) {
  const float d = *dot, iv = *inv_v, is = 1.f / *sigma;
  const long long n = (long long)rows * cols, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int r = (int)(i / cols), c = (int)(i % cols);
    g[i] = (g[i] - d * (v_raw[r] * iv) * u_hat[c]) * is;
  }
}

extern "C" int sg_dot(sg_ctx* ctx, const float* a, const float* b, long long n, float* out, int accumulate);

extern "C" int sg_spectral_norm_bwd(sg_ctx* ctx, float* g, const float* w_sn, int rows, int cols, const float* u_hat,
                                    const float* sigma, const float* fwd_scratch, float* dot_scratch) {
  SG_REQUIRE(ctx && g && w_sn && u_hat && sigma && fwd_scratch && dot_scratch && rows > 0 && cols > 0, "sg_spectral_norm_bwd: bad args");
  int rc = sg_dot(ctx, g, w_sn, (long long)rows * cols, dot_scratch, 0);
  if (rc != SG_OK) return rc;
  long long n = (long long)rows * cols;
  long long need = (n + 255) / 256, cap = (long long)ctx->num_sms * 8;
  sg_launch(ctx, k_sn_bwd, (int)(need < cap ? need : cap), 256, 0, g, dot_scratch, fwd_scratch, fwd_scratch + rows + cols, u_hat, sigma, rows,
                                                                      cols);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}
