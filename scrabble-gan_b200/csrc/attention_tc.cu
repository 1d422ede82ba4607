// Non-local block core on the tensor cores (speed mode: bf16 operands for P.V, tf32 for theta.phi^T; fp32 softmax).
// Reference: arch_ops.py:51-61   attn = softmax(theta @ phi^T) (no scaling);  o = attn @ g.
//
// Head dims are dk = 8, dv = 32, so the natural tensor-core shapes are warp-level ones: S = theta.phi^T is ONE
// mma.m16n8k8 (tf32, K = dk = 8 exactly, no padding) per 16 queries x 8 keys, and the accumulator fragments of two such
// tiles ARE the A fragment of a bf16 m16n8k16 for P.V (flash-attention-2 register chaining), so the q x kv map never
// leaves registers.  tcgen05 does not fit here: its minimum tile is M = 64/128 with K >= 8 per instruction and the
// softmax between the two GEMMs would have to round-trip TMEM; this op is < 2% of the step's FLOPs and is bounded by
// the softmax ALU work once the two GEMMs are on the tensor pipe.
//   forward      grid (ceil(Q/128), n), 8 warps x 16 queries; the image's K (tf32, transposed) and V (bf16, transposed)
//                are staged once per block in shared memory; online softmax over chunks of 64 keys
//   backward-q   same geometry: dtheta = dS . phi,  dS = P o (dO.g^T - D)
//   backward-kv  keys as the M dimension (S^T = phi.theta^T), queries streamed through shared memory in chunks of 128:
//                dg = P^T . dO,  dphi = dS^T . theta            (no atomics: one block owns its 128 keys)
//   D = rowsum(dO o O) is computed once by k_attn_rowdot.
// The exact-fp32 FFMA kernels of attention.cu remain the parity ("fp32" mode) path.
#include "common.cuh"

#define ATC_DK 8
#define ATC_DV 32
#define ATC_WARPS 8
#define ATC_THREADS (ATC_WARPS * 32)
#define ATC_ROWS (ATC_WARPS * 16)      // queries (or keys) per block

__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void mma_tf32_16x8x8(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_bf16_16x8x16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                                 uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// padded row length (elements) such that rows of 32-bit words AND rows of bf16 pairs hit distinct banks for the
// fragment access patterns used below:  len == 8 (mod 64)
static inline int atc_pad(int n) { return (n + 63) / 64 * 64 + 8; }

// D[row] = sum_j dO[row,j] * O[row,j]   (32 columns); 8 threads per row
__global__ void __launch_bounds__(256) k_attn_rowdot(const float* __restrict__ d_o, const float* __restrict__ o, long long rows,
                                                      float* __restrict__ D) {
  long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  long long row = i >> 3;
  int sub = (int)(i & 7);
  float acc = 0.f;
  if (row < rows) {
    float4 a = sg_ld4(d_o + row * ATC_DV + 4 * sub), b = sg_ld4(o + row * ATC_DV + 4 * sub);
    acc = a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  if (row < rows && sub == 0) D[row] = acc;
}

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ATC_THREADS) k_attn_fwd_tc(const float* __restrict__ theta, const float* __restrict__ phi,
                                                              const float* __restrict__ gv, int Q, int KV, int KVp,
                                                              float* __restrict__ o, float* __restrict__ lse, int kv_w,
                                                              const int* __restrict__ kv_cols) {
  // ragged batches: kv_cols[n] (may be NULL) = valid key COLUMNS of image n; key j sits in column j % kv_w
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t* Kt = reinterpret_cast<uint32_t*>(smem);                         // [8][KVp]  tf32
  __nv_bfloat16* Vt = reinterpret_cast<__nv_bfloat16*>(Kt + ATC_DK * KVp);  // [32][KVp] bf16
  const int n = blockIdx.y;
  const int vcn = kv_cols ? kv_cols[n] : kv_w;
  const int KVr = (KV + 15) & ~15;
  const float* phin = phi + (long long)n * KV * ATC_DK;
  const float* gn = gv + (long long)n * KV * ATC_DV;
  for (int i = threadIdx.x; i < KVr * ATC_DK; i += ATC_THREADS) {
    int key = i >> 3, d = i & 7;
    Kt[d * KVp + key] = key < KV ? to_tf32(phin[i]) : 0u;
  }
  for (int i = threadIdx.x; i < KVr * ATC_DV; i += ATC_THREADS) {
    int key = i >> 5, d = i & 31;
    Vt[d * KVp + key] = __float2bfloat16_rn(key < KV ? gn[i] : 0.f);
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int q0 = blockIdx.x * ATC_ROWS + warp * 16;
  if (q0 >= Q) return;
  const int ra = q0 + g, rb = q0 + g + 8;
  const float* th = theta + (long long)n * Q * ATC_DK;
  uint32_t qa[4];
  {
    int ca = ra < Q ? ra : Q - 1, cb = rb < Q ? rb : Q - 1;
    qa[0] = to_tf32(th[(long long)ca * ATC_DK + t]);
    qa[1] = to_tf32(th[(long long)cb * ATC_DK + t]);
    qa[2] = to_tf32(th[(long long)ca * ATC_DK + t + 4]);
    qa[3] = to_tf32(th[(long long)cb * ATC_DK + t + 4]);
  }
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float ma = -INFINITY, mb = -INFINITY, la = 0.f, lb = 0.f;

  for (int kc = 0; kc < KVr; kc += 64) {
    const int nj = (KVr - kc) >= 64 ? 8 : (KVr - kc) >> 3;      // n-tiles of 8 keys in this chunk (even)
    float s[8][4];
    float cma = -INFINITY, cmb = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < nj) {
        const int key0 = kc + 8 * j;
        s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
        mma_tf32_16x8x8(s[j], qa, Kt[t * KVp + key0 + g], Kt[(t + 4) * KVp + key0 + g]);
        if (key0 + 8 > KV || kv_cols) {
          const int ka = key0 + 2 * t, kb = ka + 1;
          if (ka >= KV || (kv_cols && ka % kv_w >= vcn)) { s[j][0] = -INFINITY; s[j][2] = -INFINITY; }
          if (kb >= KV || (kv_cols && kb % kv_w >= vcn)) { s[j][1] = -INFINITY; s[j][3] = -INFINITY; }
        }
        cma = fmaxf(cma, fmaxf(s[j][0], s[j][1]));
        cmb = fmaxf(cmb, fmaxf(s[j][2], s[j][3]));
      }
    }
    cma = quad_max(cma);
    cmb = quad_max(cmb);
    const float na = fmaxf(ma, cma), nb = fmaxf(mb, cmb);
    const float sa = __expf(ma - na), sb = __expf(mb - nb);     // exp(-inf) = 0 on the first chunk
    ma = na; mb = nb;
    la *= sa; lb *= sb;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) { acc[nt][0] *= sa; acc[nt][1] *= sa; acc[nt][2] *= sb; acc[nt][3] *= sb; }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < nj) {
        s[j][0] = __expf(s[j][0] - na); s[j][1] = __expf(s[j][1] - na);
        s[j][2] = __expf(s[j][2] - nb); s[j][3] = __expf(s[j][3] - nb);
        la += s[j][0] + s[j][1];
        lb += s[j][2] + s[j][3];
      }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      if (2 * jj < nj) {
        const uint32_t a0 = pack_bf16(s[2 * jj][0], s[2 * jj][1]), a1 = pack_bf16(s[2 * jj][2], s[2 * jj][3]);
        const uint32_t a2 = pack_bf16(s[2 * jj + 1][0], s[2 * jj + 1][1]), a3 = pack_bf16(s[2 * jj + 1][2], s[2 * jj + 1][3]);
        const int key0 = kc + 16 * jj;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const __nv_bfloat16* vp = Vt + (8 * nt + g) * KVp + key0 + 2 * t;
          mma_bf16_16x8x16(acc[nt], a0, a1, a2, a3, *reinterpret_cast<const uint32_t*>(vp), *reinterpret_cast<const uint32_t*>(vp + 8));
        }
      }
    }
  }
  la = quad_sum(la);
  lb = quad_sum(lb);
  const float ia = 1.f / la, ib = 1.f / lb;
  float* on = o + (long long)n * Q * ATC_DV;
  if (ra < Q) {
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
      *reinterpret_cast<float2*>(on + (long long)ra * ATC_DV + 8 * nt + 2 * t) = make_float2(acc[nt][0] * ia, acc[nt][1] * ia);
    if (t == 0) lse[(long long)n * Q + ra] = ma + __logf(la);
  }
  if (rb < Q) {
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
      *reinterpret_cast<float2*>(on + (long long)rb * ATC_DV + 8 * nt + 2 * t) = make_float2(acc[nt][2] * ib, acc[nt][3] * ib);
    if (t == 0) lse[(long long)n * Q + rb] = mb + __logf(lb);
  }
}

// ---------------------------------------------------------------------------------------------------
// backward, query side: dtheta[q] = sum_k dS[q,k] phi[k],  dS = P o (dO.g^T - D)
// smem: Kt tf32 [8][KVp] (S), Ktb bf16 [8][KVp] (dQ B operand), Vs bf16 [KV][40] (dP B operand)
// ---------------------------------------------------------------------------------------------------
#define ATC_VROW 40
__global__ void __launch_bounds__(ATC_THREADS) k_attn_bwd_q_tc(const float* __restrict__ theta, const float* __restrict__ phi,
                                                                const float* __restrict__ gv, const float* __restrict__ lse,
                                                                const float* __restrict__ d_o, const float* __restrict__ Dv, int Q,
                                                                int KV, int KVp, float* __restrict__ dtheta) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t* Kt = reinterpret_cast<uint32_t*>(smem);                               // [8][KVp] tf32
  __nv_bfloat16* Ktb = reinterpret_cast<__nv_bfloat16*>(Kt + ATC_DK * KVp);       // [8][KVp] bf16
  __nv_bfloat16* Vs = Ktb + ATC_DK * KVp;                                         // [KVr][40] bf16
  const int n = blockIdx.y;
  const int KVr = (KV + 15) & ~15;
  const float* phin = phi + (long long)n * KV * ATC_DK;
  const float* gn = gv + (long long)n * KV * ATC_DV;
  for (int i = threadIdx.x; i < KVr * ATC_DK; i += ATC_THREADS) {
    int key = i >> 3, d = i & 7;
    float v = key < KV ? phin[i] : 0.f;
    Kt[d * KVp + key] = to_tf32(v);
    Ktb[d * KVp + key] = __float2bfloat16_rn(v);
  }
  for (int i = threadIdx.x; i < KVr * ATC_DV; i += ATC_THREADS) {
    int key = i >> 5, d = i & 31;
    Vs[key * ATC_VROW + d] = __float2bfloat16_rn(key < KV ? gn[i] : 0.f);
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int q0 = blockIdx.x * ATC_ROWS + warp * 16;
  if (q0 >= Q) return;
  const int ra = q0 + g, rb = q0 + g + 8;
  const int ca = ra < Q ? ra : Q - 1, cb = rb < Q ? rb : Q - 1;
  const long long rowa = (long long)n * Q + ca, rowb = (long long)n * Q + cb;
  uint32_t qa[4];
  qa[0] = to_tf32(theta[rowa * ATC_DK + t]);
  qa[1] = to_tf32(theta[rowb * ATC_DK + t]);
  qa[2] = to_tf32(theta[rowa * ATC_DK + t + 4]);
  qa[3] = to_tf32(theta[rowb * ATC_DK + t + 4]);
  // dO as the A operand of dP = dO . V^T (16 queries x 32 dv): two k16 steps
  uint32_t da[2][4];
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    const float* pa = d_o + rowa * ATC_DV + 16 * ks + 2 * t;
    const float* pb = d_o + rowb * ATC_DV + 16 * ks + 2 * t;
    da[ks][0] = pack_bf16(pa[0], pa[1]);
    da[ks][1] = pack_bf16(pb[0], pb[1]);
    da[ks][2] = pack_bf16(pa[8], pa[9]);
    da[ks][3] = pack_bf16(pb[8], pb[9]);
  }
  const float La = lse[rowa], Lb = lse[rowb], Da = Dv[rowa], Db = Dv[rowb];
  float dq[4] = {0.f, 0.f, 0.f, 0.f};

  for (int k0 = 0; k0 < KVr; k0 += 16) {
    float ds[2][4];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int key0 = k0 + 8 * j;
      float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
      mma_tf32_16x8x8(s, qa, Kt[t * KVp + key0 + g], Kt[(t + 4) * KVp + key0 + g]);
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        const __nv_bfloat16* vp = Vs + (key0 + g) * ATC_VROW + 16 * ks + 2 * t;
        mma_bf16_16x8x16(dp, da[ks][0], da[ks][1], da[ks][2], da[ks][3], *reinterpret_cast<const uint32_t*>(vp),
                         *reinterpret_cast<const uint32_t*>(vp + 8));
      }
      const bool v0 = key0 + 2 * t < KV, v1 = key0 + 2 * t + 1 < KV;
      ds[j][0] = v0 ? __expf(s[0] - La) * (dp[0] - Da) : 0.f;
      ds[j][1] = v1 ? __expf(s[1] - La) * (dp[1] - Da) : 0.f;
      ds[j][2] = v0 ? __expf(s[2] - Lb) * (dp[2] - Db) : 0.f;
      ds[j][3] = v1 ? __expf(s[3] - Lb) * (dp[3] - Db) : 0.f;
    }
    // dQ (16 x 8 dk) += dS (16 x 16 keys) . K (16 keys x 8 dk):  B[k = key][n = dk] from Ktb[dk][key]
    const __nv_bfloat16* kp = Ktb + g * KVp + k0 + 2 * t;
    mma_bf16_16x8x16(dq, pack_bf16(ds[0][0], ds[0][1]), pack_bf16(ds[0][2], ds[0][3]), pack_bf16(ds[1][0], ds[1][1]),
                     pack_bf16(ds[1][2], ds[1][3]), *reinterpret_cast<const uint32_t*>(kp), *reinterpret_cast<const uint32_t*>(kp + 8));
  }
  if (ra < Q) *reinterpret_cast<float2*>(dtheta + ((long long)n * Q + ra) * ATC_DK + 2 * t) = make_float2(dq[0], dq[1]);
  if (rb < Q) *reinterpret_cast<float2*>(dtheta + ((long long)n * Q + rb) * ATC_DK + 2 * t) = make_float2(dq[2], dq[3]);
}

// ---------------------------------------------------------------------------------------------------
// backward, key/value side (keys are the M dimension):  dg = P^T . dO,  dphi = dS^T . theta
// per chunk of 128 queries in smem: Qt tf32 [8][QP] (S^T B operand), Qtb bf16 [8][QP] (dK B operand),
// dOs bf16 [128][40] (dP^T B operand), dOt bf16 [32][QP] (dV B operand), lse[128], D[128]
// ---------------------------------------------------------------------------------------------------
#define ATC_QC 128
#define ATC_QP 136       // 128 + 8
__global__ void __launch_bounds__(ATC_THREADS) k_attn_bwd_kv_tc(const float* __restrict__ theta, const float* __restrict__ phi,
                                                                 const float* __restrict__ gv, const float* __restrict__ lse,
                                                                 const float* __restrict__ d_o, const float* __restrict__ Dv, int Q,
                                                                 int KV, float* __restrict__ dphi, float* __restrict__ dg) {
  __shared__ uint32_t Qt[ATC_DK * ATC_QP];
  __shared__ __align__(16) __nv_bfloat16 Qtb[ATC_DK * ATC_QP];
  __shared__ __align__(16) __nv_bfloat16 dOs[ATC_QC * ATC_VROW];
  __shared__ __align__(16) __nv_bfloat16 dOt[ATC_DV * ATC_QP];
  __shared__ float Ls[ATC_QC], Ds[ATC_QC];
  const int n = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int key0 = blockIdx.x * ATC_ROWS + warp * 16;
  const bool live = key0 < KV;                       // warps beyond KV still help with the staging loads
  const int ka = key0 + g, kb = key0 + g + 8;
  const int cka = ka < KV ? ka : KV - 1, ckb = kb < KV ? kb : KV - 1;
  const long long krowa = (long long)n * KV + cka, krowb = (long long)n * KV + ckb;
  // K tile as A operand of S^T (tf32), V tile as A operand of dP^T = V . dO^T (bf16, two k16 steps over dv)
  uint32_t kfa[4], va[2][4];
  kfa[0] = to_tf32(phi[krowa * ATC_DK + t]);
  kfa[1] = to_tf32(phi[krowb * ATC_DK + t]);
  kfa[2] = to_tf32(phi[krowa * ATC_DK + t + 4]);
  kfa[3] = to_tf32(phi[krowb * ATC_DK + t + 4]);
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    const float* pa = gv + krowa * ATC_DV + 16 * ks + 2 * t;
    const float* pb = gv + krowb * ATC_DV + 16 * ks + 2 * t;
    va[ks][0] = pack_bf16(pa[0], pa[1]);
    va[ks][1] = pack_bf16(pb[0], pb[1]);
    va[ks][2] = pack_bf16(pa[8], pa[9]);
    va[ks][3] = pack_bf16(pb[8], pb[9]);
  }
  float dk[4] = {0.f, 0.f, 0.f, 0.f};
  float dv[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) dv[i][j] = 0.f;

  const float* thn = theta + (long long)n * Q * ATC_DK;
  const float* don = d_o + (long long)n * Q * ATC_DV;
  for (int qc = 0; qc < Q; qc += ATC_QC) {
    const int cnt = Q - qc < ATC_QC ? Q - qc : ATC_QC;
    __syncthreads();
    for (int i = threadIdx.x; i < ATC_QC * ATC_DK; i += ATC_THREADS) {
      int q = i >> 3, d = i & 7;
      float v = q < cnt ? thn[(long long)(qc + q) * ATC_DK + d] : 0.f;
      Qt[d * ATC_QP + q] = to_tf32(v);
      Qtb[d * ATC_QP + q] = __float2bfloat16_rn(v);
    }
    for (int i = threadIdx.x; i < ATC_QC * ATC_DV; i += ATC_THREADS) {
      int q = i >> 5, d = i & 31;
      __nv_bfloat16 v = __float2bfloat16_rn(q < cnt ? don[(long long)(qc + q) * ATC_DV + d] : 0.f);
      dOs[q * ATC_VROW + d] = v;
      dOt[d * ATC_QP + q] = v;
    }
    for (int i = threadIdx.x; i < ATC_QC; i += ATC_THREADS) {
      Ls[i] = i < cnt ? lse[(long long)n * Q + qc + i] : 0.f;
      Ds[i] = i < cnt ? Dv[(long long)n * Q + qc + i] : 0.f;
    }
    __syncthreads();
    if (!live) continue;
    const int qr = (cnt + 15) & ~15;
    for (int q0 = 0; q0 < qr; q0 += 16) {
      float pt[2][4], dst[2][4];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int qq = q0 + 8 * j;                   // 8 queries = the N dimension of this tile
        float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
        mma_tf32_16x8x8(s, kfa, Qt[t * ATC_QP + qq + g], Qt[(t + 4) * ATC_QP + qq + g]);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          const __nv_bfloat16* bp = dOs + (qq + g) * ATC_VROW + 16 * ks + 2 * t;
          mma_bf16_16x8x16(dp, va[ks][0], va[ks][1], va[ks][2], va[ks][3], *reinterpret_cast<const uint32_t*>(bp),
                           *reinterpret_cast<const uint32_t*>(bp + 8));
        }
        const int c0 = qq + 2 * t, c1 = c0 + 1;      // query columns of this thread
        const bool v0 = c0 < cnt, v1 = c1 < cnt;
        const float l0 = Ls[c0], l1 = Ls[c1], d0 = Ds[c0], d1 = Ds[c1];
        pt[j][0] = v0 ? __expf(s[0] - l0) : 0.f;
        pt[j][1] = v1 ? __expf(s[1] - l1) : 0.f;
        pt[j][2] = v0 ? __expf(s[2] - l0) : 0.f;
        pt[j][3] = v1 ? __expf(s[3] - l1) : 0.f;
        dst[j][0] = pt[j][0] * (dp[0] - d0);
        dst[j][1] = pt[j][1] * (dp[1] - d1);
        dst[j][2] = pt[j][2] * (dp[2] - d0);
        dst[j][3] = pt[j][3] * (dp[3] - d1);
      }
      const uint32_t p0 = pack_bf16(pt[0][0], pt[0][1]), p1 = pack_bf16(pt[0][2], pt[0][3]), p2 = pack_bf16(pt[1][0], pt[1][1]),
                     p3 = pack_bf16(pt[1][2], pt[1][3]);
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {               // dV (16 keys x 32 dv) += P^T (16 x 16 q) . dO (16 q x 8 dv)
        const __nv_bfloat16* bp = dOt + (8 * nt + g) * ATC_QP + q0 + 2 * t;
        mma_bf16_16x8x16(dv[nt], p0, p1, p2, p3, *reinterpret_cast<const uint32_t*>(bp), *reinterpret_cast<const uint32_t*>(bp + 8));
      }
      const __nv_bfloat16* qp = Qtb + g * ATC_QP + q0 + 2 * t;   // dK (16 keys x 8 dk) += dS^T (16 x 16 q) . Q (16 q x 8 dk)
      mma_bf16_16x8x16(dk, pack_bf16(dst[0][0], dst[0][1]), pack_bf16(dst[0][2], dst[0][3]), pack_bf16(dst[1][0], dst[1][1]),
                       pack_bf16(dst[1][2], dst[1][3]), *reinterpret_cast<const uint32_t*>(qp), *reinterpret_cast<const uint32_t*>(qp + 8));
    }
  }
  if (!live) return;
  if (ka < KV) {
    *reinterpret_cast<float2*>(dphi + ((long long)n * KV + ka) * ATC_DK + 2 * t) = make_float2(dk[0], dk[1]);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
      *reinterpret_cast<float2*>(dg + ((long long)n * KV + ka) * ATC_DV + 8 * nt + 2 * t) = make_float2(dv[nt][0], dv[nt][1]);
  }
  if (kb < KV) {
    *reinterpret_cast<float2*>(dphi + ((long long)n * KV + kb) * ATC_DK + 2 * t) = make_float2(dk[2], dk[3]);
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
      *reinterpret_cast<float2*>(dg + ((long long)n * KV + kb) * ATC_DV + 8 * nt + 2 * t) = make_float2(dv[nt][2], dv[nt][3]);
  }
}

extern "C" {

// largest KV whose K/V tiles fit the shared memory of the forward / backward-q kernels
int sg_attn_tc_supported(int q, int kv, int dk, int dv) {
  if (dk != ATC_DK || dv != ATC_DV || q < 1 || kv < 1) return 0;
  int kvp = atc_pad(kv), kvr = (kv + 15) & ~15;
  size_t bq = (size_t)ATC_DK * kvp * 4 + (size_t)ATC_DK * kvp * 2 + (size_t)kvr * ATC_VROW * 2;
  return bq <= 200 * 1024;
}

int sg_attn_fwd_tc(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv, int dk, int dv,
                   float* o, float* lse) {
  SG_REQUIRE(ctx && theta && phi && g && o && lse, "sg_attn_fwd_tc: NULL");
  SG_REQUIRE(sg_attn_tc_supported(q, kv, dk, dv), "sg_attn_fwd_tc: unsupported sizes q=%d kv=%d dk=%d dv=%d", q, kv, dk, dv);
  if (n == 0) return SG_OK;
  int kvp = atc_pad(kv);
  size_t smem = (size_t)ATC_DK * kvp * 4 + (size_t)ATC_DV * kvp * 2;
  SG_CHECK_CUDA(cudaFuncSetAttribute(k_attn_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(sg_div_up(q, ATC_ROWS), n);
  sg_launch(ctx, k_attn_fwd_tc, grid, ATC_THREADS, smem, theta, phi, g, q, kv, kvp, o, lse, kv, nullptr);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_attn_fwd_tc_masked(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv, int dk, int dv,
                          int kv_w, const int* kv_cols, float* o, float* lse) {
  SG_REQUIRE(ctx && theta && phi && g && o && lse && kv_cols, "sg_attn_fwd_tc_masked: NULL");
  SG_REQUIRE(sg_attn_tc_supported(q, kv, dk, dv) && kv_w > 0 && kv % kv_w == 0, "sg_attn_fwd_tc_masked: unsupported sizes q=%d kv=%d kv_w=%d", q, kv, kv_w);
  if (n == 0) return SG_OK;
  int kvp = atc_pad(kv);
  size_t smem = (size_t)ATC_DK * kvp * 4 + (size_t)ATC_DV * kvp * 2;
  SG_CHECK_CUDA(cudaFuncSetAttribute(k_attn_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(sg_div_up(q, ATC_ROWS), n);
  sg_launch(ctx, k_attn_fwd_tc, grid, ATC_THREADS, smem, theta, phi, g, q, kv, kvp, o, lse, kv_w, kv_cols);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_attn_bwd_tc(sg_ctx* ctx, const float* theta, const float* phi, const float* g, const float* o, const float* lse,
                   const float* d_o, int n, int q, int kv, int dk, int dv, float* dtheta, float* dphi, float* dg,
                   float* scratch /* n*q floats */) {
  SG_REQUIRE(ctx && theta && phi && g && o && lse && d_o && dtheta && dphi && dg && scratch, "sg_attn_bwd_tc: NULL");
  SG_REQUIRE(sg_attn_tc_supported(q, kv, dk, dv), "sg_attn_bwd_tc: unsupported sizes q=%d kv=%d dk=%d dv=%d", q, kv, dk, dv);
  if (n == 0) return SG_OK;
  long long rows = (long long)n * q;
  sg_launch(ctx, k_attn_rowdot, sg_div_up(rows * 8, 256), 256, 0, d_o, o, rows, scratch);
  SG_POST_LAUNCH(ctx);
  int kvp = atc_pad(kv), kvr = (kv + 15) & ~15;
  size_t smem = (size_t)ATC_DK * kvp * 4 + (size_t)ATC_DK * kvp * 2 + (size_t)kvr * ATC_VROW * 2;
  SG_CHECK_CUDA(cudaFuncSetAttribute(k_attn_bwd_q_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 gq(sg_div_up(q, ATC_ROWS), n);
  sg_launch(ctx, k_attn_bwd_q_tc, gq, ATC_THREADS, smem, theta, phi, g, lse, d_o, scratch, q, kv, kvp, dtheta);
  SG_POST_LAUNCH(ctx);
  dim3 gk(sg_div_up(kv, ATC_ROWS), n);
  sg_launch(ctx, k_attn_bwd_kv_tc, gk, ATC_THREADS, 0, theta, phi, g, lse, d_o, scratch, q, kv, dphi, dg);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
