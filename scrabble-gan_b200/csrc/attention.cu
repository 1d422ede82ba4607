// Non-local block core (K12).  Reference: arch_ops.py:51-61
//     attn = softmax(theta @ phi^T)  (over the key axis, NO 1/sqrt(d) scaling);  o = attn @ g
// theta [n,q,8], phi [n,kv,8], g [n,kv,32] fp32.  Flash-style: the q x kv map (up to 5120 x 1280 per image,
// 1.7 GB per batch in the reference) is never materialised; forward keeps only logsumexp per query.
// Head dims 8 / 32 are far too small for tensor cores to pay (K=8), so this is an FFMA kernel whose K/V tiles
// are staged in shared memory and broadcast-read as float4.
#include "common.cuh"

#define AT_DK 8
#define AT_DV 32
#define AT_KC 32      // keys per register chunk
#define AT_THREADS 128

// ---------------------------------------------------------------------------------------------------
// forward: one thread per query, block = 128 queries of one image; K/V streamed through smem in tiles of 128
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(AT_THREADS) k_attn_fwd(const float* __restrict__ theta, const float* __restrict__ phi,
                                                          const float* __restrict__ g, int Q, int KV,
                                                          float* __restrict__ o, float* __restrict__ lse, int kv_w,
                                                          const int* __restrict__ kv_cols) {
  // ragged batches: kv_cols[n] (may be NULL) = number of valid key COLUMNS of image n; key j sits in column j % kv_w
  __shared__ __align__(16) float ks[128 * AT_DK];
  __shared__ __align__(16) float vs[128 * AT_DV];
  const int n = blockIdx.y;
  const int qi = blockIdx.x * AT_THREADS + threadIdx.x;
  const bool valid = qi < Q;
  const int vcn = kv_cols ? kv_cols[n] : kv_w;
  float qv[AT_DK];
  {
    const float* tp = theta + ((long long)n * Q + (valid ? qi : 0)) * AT_DK;
    float4 a = sg_ld4(tp), b = sg_ld4(tp + 4);
    qv[0] = a.x; qv[1] = a.y; qv[2] = a.z; qv[3] = a.w; qv[4] = b.x; qv[5] = b.y; qv[6] = b.z; qv[7] = b.w;
  }
  float m = -INFINITY, l = 0.f;
  float acc[AT_DV];
#pragma unroll
  for (int j = 0; j < AT_DV; ++j) acc[j] = 0.f;

  for (int k0 = 0; k0 < KV; k0 += 128) {
    int cnt = KV - k0 < 128 ? KV - k0 : 128;
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * AT_DK / 4; i += AT_THREADS)
      reinterpret_cast<float4*>(ks)[i] = sg_ld4(phi + ((long long)n * KV + k0) * AT_DK + 4 * i);
    for (int i = threadIdx.x; i < cnt * AT_DV / 4; i += AT_THREADS)
      reinterpret_cast<float4*>(vs)[i] = sg_ld4(g + ((long long)n * KV + k0) * AT_DV + 4 * i);
    __syncthreads();
    for (int c0 = 0; c0 < cnt; c0 += AT_KC) {
      int cc = cnt - c0 < AT_KC ? cnt - c0 : AT_KC;
      float s[AT_KC];
      float cmax = -INFINITY;
#pragma unroll
      for (int i = 0; i < AT_KC; ++i) {
        if (i < cc) {
          float4 a = reinterpret_cast<const float4*>(ks)[(c0 + i) * 2], b = reinterpret_cast<const float4*>(ks)[(c0 + i) * 2 + 1];
          float d = qv[0] * a.x + qv[1] * a.y + qv[2] * a.z + qv[3] * a.w + qv[4] * b.x + qv[5] * b.y + qv[6] * b.z + qv[7] * b.w;
          if (kv_cols && (k0 + c0 + i) % kv_w >= vcn) d = -INFINITY;      // key beyond this word's width
          s[i] = d;
          cmax = fmaxf(cmax, d);
        } else {
          s[i] = -INFINITY;
        }
      }
      float mnew = fmaxf(m, cmax);
      float scale = __expf(m - mnew);      // m = -inf on the first chunk -> 0
      l *= scale;
#pragma unroll
      for (int j = 0; j < AT_DV; ++j) acc[j] *= scale;
#pragma unroll
      for (int i = 0; i < AT_KC; ++i) {
        if (i < cc) {
          float p = __expf(s[i] - mnew);
          l += p;
          const float4* vp = reinterpret_cast<const float4*>(vs) + (c0 + i) * (AT_DV / 4);
#pragma unroll
          for (int j = 0; j < AT_DV / 4; ++j) {
            float4 vv = vp[j];
            acc[4 * j + 0] = fmaf(p, vv.x, acc[4 * j + 0]);
            acc[4 * j + 1] = fmaf(p, vv.y, acc[4 * j + 1]);
            acc[4 * j + 2] = fmaf(p, vv.z, acc[4 * j + 2]);
            acc[4 * j + 3] = fmaf(p, vv.w, acc[4 * j + 3]);
          }
        }
      }
      m = mnew;
    }
  }
  if (valid) {
    float inv = 1.f / l;
    float* op = o + ((long long)n * Q + qi) * AT_DV;
#pragma unroll
    for (int j = 0; j < AT_DV / 4; ++j)
      sg_st4(op + 4 * j, make_float4(acc[4 * j] * inv, acc[4 * j + 1] * inv, acc[4 * j + 2] * inv, acc[4 * j + 3] * inv));
    lse[(long long)n * Q + qi] = m + __logf(l);
  }
}

// ---------------------------------------------------------------------------------------------------
// backward, query side: dtheta[q] = sum_kv ds * phi[kv],  ds = p * (dO.v - D),  D = dO.O,  p = exp(s - lse)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(AT_THREADS) k_attn_bwd_q(const float* __restrict__ theta, const float* __restrict__ phi,
                                                            const float* __restrict__ g, const float* __restrict__ o,
                                                            const float* __restrict__ lse, const float* __restrict__ d_o,
                                                            int Q, int KV, float* __restrict__ dtheta) {
  __shared__ __align__(16) float ks[128 * AT_DK];
  __shared__ __align__(16) float vs[128 * AT_DV];
  const int n = blockIdx.y;
  const int qi = blockIdx.x * AT_THREADS + threadIdx.x;
  const bool valid = qi < Q;
  const long long row = (long long)n * Q + (valid ? qi : 0);
  float qv[AT_DK], dov[AT_DV], dq[AT_DK];
  {
    float4 a = sg_ld4(theta + row * AT_DK), b = sg_ld4(theta + row * AT_DK + 4);
    qv[0] = a.x; qv[1] = a.y; qv[2] = a.z; qv[3] = a.w; qv[4] = b.x; qv[5] = b.y; qv[6] = b.z; qv[7] = b.w;
  }
  float D = 0.f;
#pragma unroll
  for (int j = 0; j < AT_DV / 4; ++j) {
    float4 a = sg_ld4(d_o + row * AT_DV + 4 * j), b = sg_ld4(o + row * AT_DV + 4 * j);
    dov[4 * j] = a.x; dov[4 * j + 1] = a.y; dov[4 * j + 2] = a.z; dov[4 * j + 3] = a.w;
    D += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
  }
  const float L = lse[row];
#pragma unroll
  for (int j = 0; j < AT_DK; ++j) dq[j] = 0.f;

  for (int k0 = 0; k0 < KV; k0 += 128) {
    int cnt = KV - k0 < 128 ? KV - k0 : 128;
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * AT_DK / 4; i += AT_THREADS)
      reinterpret_cast<float4*>(ks)[i] = sg_ld4(phi + ((long long)n * KV + k0) * AT_DK + 4 * i);
    for (int i = threadIdx.x; i < cnt * AT_DV / 4; i += AT_THREADS)
      reinterpret_cast<float4*>(vs)[i] = sg_ld4(g + ((long long)n * KV + k0) * AT_DV + 4 * i);
    __syncthreads();
    for (int i = 0; i < cnt; ++i) {
      float4 a = reinterpret_cast<const float4*>(ks)[i * 2], b = reinterpret_cast<const float4*>(ks)[i * 2 + 1];
      float s = qv[0] * a.x + qv[1] * a.y + qv[2] * a.z + qv[3] * a.w + qv[4] * b.x + qv[5] * b.y + qv[6] * b.z + qv[7] * b.w;
      float p = __expf(s - L);
      float dp = 0.f;
      const float4* vp = reinterpret_cast<const float4*>(vs) + i * (AT_DV / 4);
#pragma unroll
      for (int j = 0; j < AT_DV / 4; ++j) {
        float4 vv = vp[j];
        dp += dov[4 * j] * vv.x + dov[4 * j + 1] * vv.y + dov[4 * j + 2] * vv.z + dov[4 * j + 3] * vv.w;
      }
      float ds = p * (dp - D);
      dq[0] = fmaf(ds, a.x, dq[0]); dq[1] = fmaf(ds, a.y, dq[1]); dq[2] = fmaf(ds, a.z, dq[2]); dq[3] = fmaf(ds, a.w, dq[3]);
      dq[4] = fmaf(ds, b.x, dq[4]); dq[5] = fmaf(ds, b.y, dq[5]); dq[6] = fmaf(ds, b.z, dq[6]); dq[7] = fmaf(ds, b.w, dq[7]);
    }
  }
  if (valid) {
    sg_st4(dtheta + row * AT_DK, make_float4(dq[0], dq[1], dq[2], dq[3]));
    sg_st4(dtheta + row * AT_DK + 4, make_float4(dq[4], dq[5], dq[6], dq[7]));
  }
}

// ---------------------------------------------------------------------------------------------------
// backward, key/value side: one thread per key; queries streamed through smem in tiles of 64.
//   dg[kv] = sum_q p * dO[q];   dphi[kv] = sum_q ds * theta[q]
// grid: (ceil(KV/128), n, q_splits); partial sums over the q-splits are combined with atomicAdd.
// ---------------------------------------------------------------------------------------------------
#define AT_QT 64
__global__ void __launch_bounds__(AT_THREADS) k_attn_bwd_kv(const float* __restrict__ theta, const float* __restrict__ phi,
                                                             const float* __restrict__ g, const float* __restrict__ o,
                                                             const float* __restrict__ lse, const float* __restrict__ d_o,
                                                             int Q, int KV, int q_per_split, float* __restrict__ dphi,
                                                             float* __restrict__ dg, unsigned int* __restrict__ sems) {
  __shared__ __align__(16) float qs[AT_QT * AT_DK];
  __shared__ __align__(16) float dos[AT_QT * AT_DV];
  __shared__ float ls[AT_QT], Ds[AT_QT];
  const int n = blockIdx.y;
  const int ki = blockIdx.x * AT_THREADS + threadIdx.x;
  const bool valid = ki < KV;
  const long long krow = (long long)n * KV + (valid ? ki : 0);
  float kv[AT_DK], vv[AT_DV], dk[AT_DK], dv[AT_DV];
  {
    float4 a = sg_ld4(phi + krow * AT_DK), b = sg_ld4(phi + krow * AT_DK + 4);
    kv[0] = a.x; kv[1] = a.y; kv[2] = a.z; kv[3] = a.w; kv[4] = b.x; kv[5] = b.y; kv[6] = b.z; kv[7] = b.w;
  }
#pragma unroll
  for (int j = 0; j < AT_DV / 4; ++j) {
    float4 a = sg_ld4(g + krow * AT_DV + 4 * j);
    vv[4 * j] = a.x; vv[4 * j + 1] = a.y; vv[4 * j + 2] = a.z; vv[4 * j + 3] = a.w;
  }
#pragma unroll
  for (int j = 0; j < AT_DK; ++j) dk[j] = 0.f;
#pragma unroll
  for (int j = 0; j < AT_DV; ++j) dv[j] = 0.f;

  const int qbeg = blockIdx.z * q_per_split;
  const int qend = qbeg + q_per_split < Q ? qbeg + q_per_split : Q;
  for (int q0 = qbeg; q0 < qend; q0 += AT_QT) {
    int cnt = qend - q0 < AT_QT ? qend - q0 : AT_QT;
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * AT_DK / 4; i += AT_THREADS)
      reinterpret_cast<float4*>(qs)[i] = sg_ld4(theta + ((long long)n * Q + q0) * AT_DK + 4 * i);
    for (int i = threadIdx.x; i < cnt * AT_DV / 4; i += AT_THREADS)
      reinterpret_cast<float4*>(dos)[i] = sg_ld4(d_o + ((long long)n * Q + q0) * AT_DV + 4 * i);
    if (threadIdx.x < cnt) {
      long long r = (long long)n * Q + q0 + threadIdx.x;
      ls[threadIdx.x] = lse[r];
      float D = 0.f;
#pragma unroll
      for (int j = 0; j < AT_DV / 4; ++j) {
        float4 a = sg_ld4(d_o + r * AT_DV + 4 * j), b = sg_ld4(o + r * AT_DV + 4 * j);
        D += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
      }
      Ds[threadIdx.x] = D;
    }
    __syncthreads();
    for (int i = 0; i < cnt; ++i) {
      float4 a = reinterpret_cast<const float4*>(qs)[i * 2], b = reinterpret_cast<const float4*>(qs)[i * 2 + 1];
      float s = kv[0] * a.x + kv[1] * a.y + kv[2] * a.z + kv[3] * a.w + kv[4] * b.x + kv[5] * b.y + kv[6] * b.z + kv[7] * b.w;
      float p = __expf(s - ls[i]);
      float dp = 0.f;
      const float4* dp4 = reinterpret_cast<const float4*>(dos) + i * (AT_DV / 4);
#pragma unroll
      for (int j = 0; j < AT_DV / 4; ++j) {
        float4 d = dp4[j];
        dp += d.x * vv[4 * j] + d.y * vv[4 * j + 1] + d.z * vv[4 * j + 2] + d.w * vv[4 * j + 3];
        dv[4 * j] = fmaf(p, d.x, dv[4 * j]);
        dv[4 * j + 1] = fmaf(p, d.y, dv[4 * j + 1]);
        dv[4 * j + 2] = fmaf(p, d.z, dv[4 * j + 2]);
        dv[4 * j + 3] = fmaf(p, d.w, dv[4 * j + 3]);
      }
      float ds = p * (dp - Ds[i]);
      dk[0] = fmaf(ds, a.x, dk[0]); dk[1] = fmaf(ds, a.y, dk[1]); dk[2] = fmaf(ds, a.z, dk[2]); dk[3] = fmaf(ds, a.w, dk[3]);
      dk[4] = fmaf(ds, b.x, dk[4]); dk[5] = fmaf(ds, b.y, dk[5]); dk[6] = fmaf(ds, b.z, dk[6]); dk[7] = fmaf(ds, b.w, dk[7]);
    }
  }
  // the q-splits of a key block add in split order (ordered turns, common.cuh scheme A): bitwise repeatable
  unsigned int* sem = sems + (long long)blockIdx.y * gridDim.x + blockIdx.x;
  if (gridDim.z > 1) {
    if (threadIdx.x == 0) sg_turn_wait(sem, blockIdx.z);
    __syncthreads();
  }
  if (valid) {
#pragma unroll
    for (int j = 0; j < AT_DK; ++j) atomicAdd(dphi + krow * AT_DK + j, dk[j]);
#pragma unroll
    for (int j = 0; j < AT_DV; ++j) atomicAdd(dg + krow * AT_DV + j, dv[j]);
  }
  if (gridDim.z > 1) {
    __syncthreads();
    if (threadIdx.x == 0) sg_turn_pass(sem, blockIdx.z, gridDim.z);
  }
}

extern "C" {

int sg_attn_fwd(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv, int dk,
                int dv, float* o, float* lse) {
  SG_REQUIRE(ctx && theta && phi && g && o && lse, "sg_attn_fwd: NULL");
  SG_REQUIRE(dk == AT_DK && dv == AT_DV, "sg_attn_fwd: only dk=8, dv=32 (C=64 non-local block) is built (got %d,%d)", dk, dv);
  SG_REQUIRE(q > 0 && kv > 0 && n >= 0, "sg_attn_fwd: bad sizes");
  if (n == 0) return SG_OK;
  dim3 grid(sg_div_up(q, AT_THREADS), n);
  sg_launch(ctx, k_attn_fwd, grid, AT_THREADS, 0, theta, phi, g, q, kv, o, lse, kv, nullptr);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

/* ragged batch (inference): key j of image n lies in column j % kv_w of the key map; columns >= kv_cols[n] are outside the word */
int sg_attn_fwd_masked(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv, int dk,
                       int dv, int kv_w, const int* kv_cols, float* o, float* lse) {
  SG_REQUIRE(ctx && theta && phi && g && o && lse && kv_cols, "sg_attn_fwd_masked: NULL");
  SG_REQUIRE(dk == AT_DK && dv == AT_DV, "sg_attn_fwd_masked: only dk=8, dv=32 is built (got %d,%d)", dk, dv);
  SG_REQUIRE(q > 0 && kv > 0 && n >= 0 && kv_w > 0 && kv % kv_w == 0, "sg_attn_fwd_masked: bad sizes");
  if (n == 0) return SG_OK;
  dim3 grid(sg_div_up(q, AT_THREADS), n);
  sg_launch(ctx, k_attn_fwd, grid, AT_THREADS, 0, theta, phi, g, q, kv, o, lse, kv_w, kv_cols);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_attn_bwd(sg_ctx* ctx, const float* theta, const float* phi, const float* g, const float* o, const float* lse,
                const float* d_o, int n, int q, int kv, int dk, int dv, float* dtheta, float* dphi, float* dg) {
  SG_REQUIRE(ctx && theta && phi && g && o && lse && d_o && dtheta && dphi && dg, "sg_attn_bwd: NULL");
  SG_REQUIRE(dk == AT_DK && dv == AT_DV, "sg_attn_bwd: only dk=8, dv=32 is built (got %d,%d)", dk, dv);
  SG_REQUIRE(q > 0 && kv > 0 && n >= 0, "sg_attn_bwd: bad sizes");
  if (n == 0) return SG_OK;
  dim3 grid(sg_div_up(q, AT_THREADS), n);
  sg_launch(ctx, k_attn_bwd_q, grid, AT_THREADS, 0, theta, phi, g, o, lse, d_o, q, kv, dtheta);
  SG_POST_LAUNCH(ctx);
  SG_CHECK_CUDA(cudaMemsetAsync(dphi, 0, sizeof(float) * (size_t)n * kv * AT_DK, ctx->stream));
  SG_CHECK_CUDA(cudaMemsetAsync(dg, 0, sizeof(float) * (size_t)n * kv * AT_DV, ctx->stream));
  int kblocks = sg_div_up(kv, AT_THREADS);
  int splits = sg_div_up(2LL * ctx->num_sms, (long long)kblocks * n);
  int max_splits = sg_div_up(q, 4 * AT_QT);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if ((long long)kblocks * n > SG_DET_TICKETS) splits = 1;
  int qps = sg_div_up(sg_div_up(q, splits), AT_QT) * AT_QT;
  splits = sg_div_up(q, qps);
  dim3 g2(kblocks, n, splits);
  sg_launch(ctx, k_attn_bwd_kv, g2, AT_THREADS, 0, theta, phi, g, o, lse, d_o, q, kv, qps, dphi, dg, ctx->det_tickets);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
