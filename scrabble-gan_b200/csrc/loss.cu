// GAN losses + ScrabbleGAN "gradient balancing" (K16, K17).
// Reference: net_loss.py:38-54 (hinge), :4-35 (not_saturating), data_utils.py:418-442 (13 means) and
// :476-490 (apply_gradient_balancing: population std of the per-sample losses, differentiable, no guards).
// The per-sample upstream weights for every backward pass are produced in closed form:
//   S = sum_i g_i + alpha (sd_g/sd_r) r_i   =>   dS/dg_i = 1 + alpha (R/sd_r)(g_i - mean_g)/(N sd_g)
//                                                dS/dr_i = alpha [ sd_g/sd_r - sd_g R (r_i - mean_r)/(N sd_r^3) ]
// Sums are kept in double and exchanged between the two kernels so that data-parallel replicas can
// all-reduce them (the std is then over the GLOBAL batch).
#include "common.cuh"

enum { SUM_G = 0, SUM_G2, SUM_R, SUM_R2, SUM_RREAL, SUM_DLR, SUM_DLF, SUM_SL1, SUM_SL2, SUM_N };

__device__ __forceinline__ float sce(float x, float z) {   // tf.nn.sigmoid_cross_entropy_with_logits
  return fmaxf(x, 0.f) - x * z + log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__device__ __forceinline__ float g_of(int kind, int use_w, float d_fake, float s_fake, float s5) {
  if (kind == SG_LOSS_HINGE) return use_w ? -(d_fake + s_fake) : -d_fake;
  return use_w ? sce(d_fake, 1.f) + sce(s5, 1.f) : sce(d_fake, 1.f);
}

__device__ double block_sum_d(double v, double* sm) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  int nw = blockDim.x >> 5;
  for (int i = 0; i < nw; ++i) r += sm[i];
  return r;
}

__global__ void k_loss_sums(int kind, int use_w, const float* d_real, const float* d_fake, const float* s_real,
                            const float* s_fake, const float* s5, const float* r_fake, const float* r_real, int b,
                            double* sums) {
  __shared__ double sm[32];
  double acc[SUM_N];
  for (int j = 0; j < SUM_N; ++j) acc[j] = 0.0;
  for (int i = threadIdx.x; i < b; i += blockDim.x) {
    float dr = d_real[i], df = d_fake[i];
    float sr = use_w ? s_real[i] : 0.f, sf = use_w ? s_fake[i] : 0.f, sx = (use_w && s5) ? s5[i] : 0.f;
    float g = g_of(kind, use_w, df, sf, sx);
    float r = r_fake[i];
    acc[SUM_G] += g;
    acc[SUM_G2] += (double)g * g;
    acc[SUM_R] += r;
    acc[SUM_R2] += (double)r * r;
    acc[SUM_RREAL] += r_real[i];
    if (kind == SG_LOSS_HINGE) {
      acc[SUM_DLR] += fmaxf(1.f - dr, 0.f);
      acc[SUM_DLF] += fmaxf(1.f + df, 0.f);
      if (use_w) { acc[SUM_SL1] += fmaxf(1.f - sr, 0.f); acc[SUM_SL2] += fmaxf(1.f + sf, 0.f); }
    } else {
      acc[SUM_DLR] += sce(dr, 1.f);
      acc[SUM_DLF] += sce(df, 0.f);
      if (use_w) { acc[SUM_SL1] += sce(sr, 1.f); acc[SUM_SL2] += sce(sf, 0.f); }
    }
  }
  for (int j = 0; j < SUM_N; ++j) {
    double t = block_sum_d(acc[j], sm);
    if (threadIdx.x == 0) sums[j] = t;
  }
  if (threadIdx.x == 0) {
    sums[SUM_N] = (double)b;
    for (int j = SUM_N + 1; j < SG_LOSS_NSUMS; ++j) sums[j] = 0.0;
  }
}

__global__ void k_loss_finish(int kind, int use_w, int balance, float alpha, const float* d_real, const float* d_fake,
                              const float* s_real, const float* s_fake, const float* s5, const float* r_fake, int b,
                              const double* sums, float* up_d_real, float* up_d_fake_d, float* up_s_real,
                              float* up_s_fake_w, float* up_s_slot5, float* up_d_fake_g, float* up_s_fake_g,
                              float* up_r_fake_g, float* stats) {
  const double N = sums[SUM_N];
  const double mean_g = sums[SUM_G] / N, mean_r = sums[SUM_R] / N;
  double var_g = sums[SUM_G2] / N - mean_g * mean_g, var_r = sums[SUM_R2] / N - mean_r * mean_r;
  if (var_g < 0) var_g = 0;
  if (var_r < 0) var_r = 0;
  const double sd_g = sqrt(var_g), sd_r = sqrt(var_r);
  const double R = sums[SUM_R];
  const double ratio = sd_g / sd_r;          // no zero guard: the reference has none (data_utils.py:488)
  for (int i = threadIdx.x; i < b; i += blockDim.x) {
    float dr = d_real[i], df = d_fake[i];
    float sr = use_w ? s_real[i] : 0.f, sf = use_w ? s_fake[i] : 0.f, sx = (use_w && s5) ? s5[i] : 0.f;
    float g = g_of(kind, use_w, df, sf, sx);
    float r = r_fake[i];
    double cg = 1.0, cr = 1.0;
    if (balance) {
      cg = 1.0 + (double)alpha * (R / sd_r) * ((double)g - mean_g) / (N * sd_g);
      cr = (double)alpha * (ratio - sd_g * R * ((double)r - mean_r) / (N * sd_r * sd_r * sd_r));
    }
    float dg_dd, dg_ds;
    if (kind == SG_LOSS_HINGE) {
      up_d_real[i] = (1.f - dr > 0.f) ? -1.f : 0.f;
      up_d_fake_d[i] = (1.f + df > 0.f) ? 1.f : 0.f;
      if (use_w) {
        up_s_real[i] = (1.f - sr > 0.f) ? -1.f : 0.f;
        up_s_fake_w[i] = (1.f + sf > 0.f) ? 1.f : 0.f;
        if (up_s_slot5) up_s_slot5[i] = 0.f;
      }
      dg_dd = -1.f;
      dg_ds = use_w ? -1.f : 0.f;
    } else {
      up_d_real[i] = sigmoidf_(dr) - 1.f;
      up_d_fake_d[i] = sigmoidf_(df);
      if (use_w) {
        up_s_real[i] = sigmoidf_(sr) - 1.f;
        up_s_fake_w[i] = sigmoidf_(sf);
        if (up_s_slot5) up_s_slot5[i] = 0.f;
      }
      dg_dd = sigmoidf_(df) - 1.f;
      dg_ds = 0.f;       // bug-compatible: g uses the 5th slot (W(real images)), not W(G(z))  (SURVEY Q1)
    }
    up_d_fake_g[i] = (float)(cg * dg_dd);
    if (use_w && up_s_fake_g) up_s_fake_g[i] = (float)(cg * dg_ds);
    up_r_fake_g[i] = (float)cr;
  }
  if (threadIdx.x == 0) {
    double mean_rreal = sums[SUM_RREAL] / N;
    double r_bal = (double)alpha * ratio * mean_r;
    double g_added = mean_g + mean_r, g_bal = mean_g + r_bal;
    double dlr = sums[SUM_DLR] / N, dlf = sums[SUM_DLF] / N, s1 = sums[SUM_SL1] / N, s2 = sums[SUM_SL2] / N;
    stats[0] = (float)mean_r;        // r_loss_fake
    stats[1] = (float)mean_rreal;    // r_loss_real
    stats[2] = (float)r_bal;         // r_loss_balanced
    stats[3] = (float)mean_g;        // g_loss
    stats[4] = (float)g_added;       // g_loss_added
    stats[5] = (float)g_bal;         // g_loss_balanced
    stats[6] = (float)(dlr + dlf);   // d_loss
    stats[7] = (float)dlr;
    stats[8] = (float)dlf;
    stats[9] = (float)(balance ? g_bal : g_added);   // g_loss_final
    stats[10] = alpha;
    stats[11] = (float)sd_r;         // r_loss_fake_std
    stats[12] = (float)sd_g;         // g_loss_std
    stats[13] = (float)(s1 + s2);    // s_loss
    stats[14] = (float)s1;
    stats[15] = (float)s2;
  }
}

extern "C" {

int sg_loss_sums(sg_ctx* ctx, int kind, int use_w, const float* d_real, const float* d_fake, const float* s_real,
                 const float* s_fake, const float* s_slot5, const float* r_fake, const float* r_real, int b,
                 double* sums) {
  SG_REQUIRE(ctx && d_real && d_fake && r_fake && r_real && sums && b > 0, "sg_loss_sums: bad args");
  SG_REQUIRE(!use_w || (s_real && s_fake), "sg_loss_sums: use_w needs s_real and s_fake");
  SG_REQUIRE(kind == SG_LOSS_HINGE || kind == SG_LOSS_NOT_SATURATING, "sg_loss_sums: bad loss kind %d", kind);
  sg_launch(ctx, k_loss_sums, 1, 256, 0, kind, use_w, d_real, d_fake, s_real, s_fake, s_slot5, r_fake, r_real, b, sums);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_loss_finish(sg_ctx* ctx, int kind, int use_w, int balance, float alpha, const float* d_real, const float* d_fake,
                   const float* s_real, const float* s_fake, const float* s_slot5, const float* r_fake, int b,
                   const double* sums, float* up_d_real, float* up_d_fake_d, float* up_s_real, float* up_s_fake_w,
                   float* up_s_slot5, float* up_d_fake_g, float* up_s_fake_g, float* up_r_fake_g, float* stats) {
  SG_REQUIRE(ctx && d_real && d_fake && r_fake && sums && up_d_real && up_d_fake_d && up_d_fake_g && up_r_fake_g && stats && b > 0,
             "sg_loss_finish: bad args");
  SG_REQUIRE(!use_w || (s_real && s_fake && up_s_real && up_s_fake_w), "sg_loss_finish: use_w needs the s_* buffers");
  SG_REQUIRE(kind == SG_LOSS_HINGE || kind == SG_LOSS_NOT_SATURATING, "sg_loss_finish: bad loss kind %d", kind);
  sg_launch(ctx, k_loss_finish, 1, 256, 0, kind, use_w, balance, alpha, d_real, d_fake, s_real, s_fake, s_slot5, r_fake, b,
                                            sums, up_d_real, up_d_fake_d, up_s_real, up_s_fake_w, up_s_slot5, up_d_fake_g,
                                            up_s_fake_g, up_r_fake_g, stats);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// stand-alone forms of the reference's public functions (used when callers invoke hinge / not_saturating /
// apply_gradient_balancing directly rather than through train_step's fused path)
// ---------------------------------------------------------------------------------------------------
// terms[7][b]: d_loss, d_loss_real, d_loss_fake, g_loss, s_loss, s_loss_1, s_loss_2   (net_loss.py return order)
__global__ void k_loss_terms(int kind, const float* d_real, const float* d_fake, const float* s_a, const float* s_b,
                             const float* s_c, int b, float* terms) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < b; i += gridDim.x * blockDim.x) {
    float dr = d_real[i], df = d_fake[i], sa = s_a[i], sb = s_b[i], sc = s_c ? s_c[i] : 0.f;
    float dlr, dlf, g, s1, s2;
    if (kind == SG_LOSS_HINGE) {
      dlr = fmaxf(1.f - dr, 0.f); dlf = fmaxf(1.f + df, 0.f);
      s1 = fmaxf(1.f - sa, 0.f); s2 = fmaxf(1.f + sb, 0.f);
      g = -(df + sb);
    } else {
      dlr = sce(dr, 1.f); dlf = sce(df, 0.f);
      s1 = sce(sa, 1.f); s2 = sce(sb, 0.f);
      g = sce(df, 1.f) + sce(sc, 1.f);
    }
    terms[0 * b + i] = dlr + dlf; terms[1 * b + i] = dlr; terms[2 * b + i] = dlf; terms[3 * b + i] = g;
    terms[4 * b + i] = s1 + s2; terms[5 * b + i] = s1; terms[6 * b + i] = s2;
  }
}

// g_bal = g + alpha (sd_g / sd_r) r ; r_bal = alpha (sd_g / sd_r) r ; stds = {sd_r, sd_g}   (single CTA)
__global__ void k_grad_balance(const float* r, const float* g, int b, float alpha, float* g_bal, float* r_bal, float* stds) {
  __shared__ double sm[32];
  double sr = 0, sr2 = 0, sg = 0, sg2 = 0;
  for (int i = threadIdx.x; i < b; i += blockDim.x) {
    double rv = r[i], gv = g[i];
    sr += rv; sr2 += rv * rv; sg += gv; sg2 += gv * gv;
  }
  sr = block_sum_d(sr, sm); sr2 = block_sum_d(sr2, sm); sg = block_sum_d(sg, sm); sg2 = block_sum_d(sg2, sm);
  double mr = sr / b, mg = sg / b;
  double vr = sr2 / b - mr * mr, vg = sg2 / b - mg * mg;
  double sdr = sqrt(vr > 0 ? vr : 0), sdg = sqrt(vg > 0 ? vg : 0);
  float ratio = (float)(sdg / sdr);
  for (int i = threadIdx.x; i < b; i += blockDim.x) {
    float rb = alpha * (ratio * r[i]);
    r_bal[i] = rb;
    g_bal[i] = g[i] + rb;
  }
  if (threadIdx.x == 0) { stds[0] = (float)sdr; stds[1] = (float)sdg; }
}

extern "C" {

int sg_loss_terms(sg_ctx* ctx, int kind, const float* d_real, const float* d_fake, const float* s_a, const float* s_b,
                  const float* s_c, int b, float* terms) {
  SG_REQUIRE(ctx && d_real && d_fake && s_a && s_b && terms && b > 0, "sg_loss_terms: bad args");
  SG_REQUIRE(kind == SG_LOSS_HINGE || kind == SG_LOSS_NOT_SATURATING, "sg_loss_terms: bad loss kind %d", kind);
  sg_launch(ctx, k_loss_terms, sg_div_up(b, 256), 256, 0, kind, d_real, d_fake, s_a, s_b, s_c, b, terms);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_grad_balance(sg_ctx* ctx, const float* r_fake, const float* g_loss, int b, float alpha, float* g_balanced,
                    float* r_balanced, float* stds) {
  SG_REQUIRE(ctx && r_fake && g_loss && g_balanced && r_balanced && stds && b > 0, "sg_grad_balance: bad args");
  sg_launch(ctx, k_grad_balance, 1, 256, 0, r_fake, g_loss, b, alpha, g_balanced, r_balanced, stds);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// Paper-faithful gradient balancing (ScrabbleGAN, arXiv 2003.10557, section 3.4; north_star "std(grad_D)/std(grad_R)"):
//     grad_R <- alpha * (std(grad_D) / std(grad_R)) * grad_R,   both gradients taken w.r.t. the generated IMAGE,
//     std = population std over every element of the (global) batch of image gradients.
// The reference fork balances LOSS values instead (data_utils.py:476-490, SURVEY Q6); this is the opt-in alternative.
// sums[0..4] = {sum gd, sum gd^2, sum gr, sum gr^2, n} in double: all-reduce them across replicas between the two calls.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_imgbal_sums(const float* __restrict__ gd, const float* __restrict__ gr, long long n,
                                                      double* __restrict__ sums, double* __restrict__ scratch, unsigned int* ticket) {
  __shared__ double sm[32];
  double a[4] = {0.0, 0.0, 0.0, 0.0};
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    double d = gd[i], r = gr[i];
    a[0] += d; a[1] += d * d; a[2] += r; a[3] += r * r;
  }
  for (int j = 0; j < 4; ++j) {
    double t = block_sum_d(a[j], sm);
    if (threadIdx.x == 0) scratch[(long long)blockIdx.x * 4 + j] = t;
  }
  if (!sg_det_arrive_last(ticket, gridDim.x)) return;        // per-block partials, added in block order by the last block
  if (threadIdx.x < 4) {
    double t = 0.0;
    for (unsigned int b = 0; b < gridDim.x; ++b) t += __ldcg(scratch + (long long)b * 4 + threadIdx.x);
    sums[threadIdx.x] = t;
  }
  if (threadIdx.x == 0) {
    sums[4] = (double)n;
    for (int j = 5; j < 8; ++j) sums[j] = 0.0;
  }
}

// out = gd + alpha (sd_d / sd_r) gr;  stats (the step's 16-tuple) is patched: r_loss_balanced = ratio * r_loss_fake,
// g_loss_balanced = g_loss_final = g_loss + r_loss_balanced, alpha, r_loss_fake_std := sd_r, g_loss_std := sd_d
__global__ void k_imgbal_apply(const float* __restrict__ gd, const float* __restrict__ gr, long long n, float alpha,
                               const double* __restrict__ sums, float* __restrict__ out, float* __restrict__ stats) {
  const double N = sums[4];
  const double md = sums[0] / N, mr = sums[2] / N;
  double vd = sums[1] / N - md * md, vr = sums[3] / N - mr * mr;
  const double sd_d = sqrt(vd > 0 ? vd : 0), sd_r = sqrt(vr > 0 ? vr : 0);
  const float ratio = (float)((double)alpha * sd_d / sd_r);          // no zero guard, as in the loss-level original
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = gd[i] + ratio * gr[i];
  if (stats && blockIdx.x == 0 && threadIdx.x == 0) {
    float r_bal = ratio * stats[0];
    stats[2] = r_bal;
    stats[5] = stats[3] + r_bal;
    stats[9] = stats[3] + r_bal;
    stats[10] = alpha;
    stats[11] = (float)sd_r;
    stats[12] = (float)sd_d;
  }
}

extern "C" {

int sg_image_grad_balance_sums(sg_ctx* ctx, const float* grad_d, const float* grad_r, long long n, double* sums) {
  SG_REQUIRE(ctx && grad_d && grad_r && sums && n > 0, "sg_image_grad_balance_sums: bad args");
  long long blocks = (n + 256 * 8 - 1) / (256 * 8), cap = (long long)ctx->num_sms * 2;
  if (blocks > cap) blocks = cap;
  sg_launch(ctx, k_imgbal_sums, (int)blocks, 256, 0, grad_d, grad_r, n, sums, reinterpret_cast<double*>(ctx->det_scratch), ctx->det_tickets);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_image_grad_balance_apply(sg_ctx* ctx, const float* grad_d, const float* grad_r, long long n, float alpha, const double* sums,
                                float* out, float* stats) {
  SG_REQUIRE(ctx && grad_d && grad_r && sums && out && n > 0, "sg_image_grad_balance_apply: bad args");
  long long blocks = (n + 255) / 256, cap = (long long)ctx->num_sms * 8;
  if (blocks > cap) blocks = cap;
  sg_launch(ctx, k_imgbal_apply, (int)blocks, 256, 0, grad_d, grad_r, n, alpha, sums, out, stats);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
