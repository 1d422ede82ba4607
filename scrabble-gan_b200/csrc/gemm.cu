// Small fp32 GEMM for the Dense layers (K14) and the attention 1x1 projections:
//   C[m,n] (+)= sum_k opA(m,k) * opB(k,n) + bias[n]      row-major, arbitrary sizes.
// Reference call sites: resnet_ops.py:18,24 (CBN gamma/beta), net_architecture.py:55,251,342,401.
// 64x64x16 shared-memory tiles, 256 threads, 4x4 register blocking.  These GEMMs are tiny (<0.1% of step
// FLOPs) or HBM-bound (K <= 64), so they stay on the FFMA pipe by design.
#include "common.cuh"

#define GT_M 64
#define GT_N 64

// GT_K = 16: generic k loop.  GT_K = 64: the whole reduction (K <= 64: CBN gamma / beta Dense layers with K = 32 or the
// batch as K) is staged in ONE round of loads -- a single global-memory latency instead of one per 16-wide k step.
template <int GT_K>
__global__ void __launch_bounds__(256) k_gemm(int ta, int tb, int M, int N, int K, const float* __restrict__ A, int lda,
                                               const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
                                               const float* __restrict__ bias, int accumulate, int k_per_split, float* __restrict__ scratch, unsigned int* __restrict__ tickets) {
  __shared__ float As[GT_K][GT_M + 4];
  __shared__ float Bs[GT_K][GT_N + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * GT_M, n0 = blockIdx.x * GT_N;
  const int tx = tid % 16, ty = tid / 16;      // thread computes rows ty*4..+3, cols tx*4..+3
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int kbeg = blockIdx.z * k_per_split;
  const int kend = (kbeg + k_per_split < K) ? kbeg + k_per_split : K;
  const bool split = gridDim.z > 1;
  for (int k0 = kbeg; k0 < kend; k0 += GT_K) {
#pragma unroll
    for (int i = 0; i < GT_K / 4; ++i) {
      int idx = tid + i * 256;
      int mm, kk;
      if (ta) { mm = idx % GT_M; kk = idx / GT_M; } else { kk = idx % GT_K; mm = idx / GT_K; }
      int gm = m0 + mm, gk = k0 + kk;
      float v = 0.f;
      if (gm < M && gk < kend) v = ta ? A[(long long)gk * lda + gm] : A[(long long)gm * lda + gk];
      As[kk][mm] = v;
    }
#pragma unroll
    for (int i = 0; i < GT_K / 4; ++i) {
      int idx = tid + i * 256;
      int nn, kk;
      if (tb) { kk = idx % GT_K; nn = idx / GT_K; } else { nn = idx % GT_N; kk = idx / GT_N; }
      int gn = n0 + nn, gk = k0 + kk;
      float v = 0.f;
      if (gn < N && gk < kend) v = tb ? B[(long long)gn * ldb + gk] : B[(long long)gk * ldb + gn];
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GT_K; ++kk) {
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
  if (!split) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int gm = m0 + ty * 4 + i;
      if (gm >= M) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int gn = n0 + tx * 4 + j;
        if (gn >= N) continue;
        float v = acc[i][j];
        if (bias) v += bias[gn];
        float* p = C + (long long)gm * ldc + gn;
        if (accumulate) v += *p;
        *p = v;
      }
    }
    return;
  }
  // split-K, deterministic (common.cuh scheme B): every split stores its 64 x 64 partial tile in its own scratch slot; the
  // last split of the tile to arrive adds the slots in split order and writes C (+ bias, + previous C when accumulating)
  const int tile = blockIdx.y * gridDim.x + blockIdx.x;
  const unsigned int nsp = gridDim.z, tk_per_tile = 1 + (nsp + SG_DET_GROUP - 1) / SG_DET_GROUP;
  const long long fl_per_tile = (long long)GT_M * GT_N * (nsp + (nsp > 32 ? (nsp + SG_DET_GROUP - 1) / SG_DET_GROUP : 0));
  float* slots = scratch + (long long)tile * fl_per_tile;
  float* mine = slots + (long long)blockIdx.z * (GT_M * GT_N);
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4*>(mine + (ty * 4 + i) * GT_N + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  sg_det_finish(slots, slots + (long long)nsp * (GT_M * GT_N), tickets + (long long)tile * tk_per_tile, nsp, blockIdx.z, GT_M * GT_N,
                [&](int idx, float t) {
                  int gm = m0 + idx / GT_N, gn = n0 + idx % GT_N;
                  if (gm >= M || gn >= N) return;
                  float* p = C + (long long)gm * ldc + gn;
                  float v = t + (bias ? bias[gn] : 0.f);
                  if (accumulate) v += *p;
                  *p = v;
                });
}

extern "C" int sg_gemm(sg_ctx* ctx, int trans_a, int trans_b, int m, int n, int k, const float* a, int lda,
                       const float* b, int ldb, float* c, int ldc, const float* bias, int accumulate) {
  SG_REQUIRE(ctx && a && b && c, "sg_gemm: NULL");
  SG_REQUIRE(m >= 0 && n >= 0 && k >= 0, "sg_gemm: negative dims");
  if (m == 0 || n == 0) return SG_OK;
  dim3 grid(sg_div_up(n, GT_N), sg_div_up(m, GT_M));
  SG_REQUIRE(grid.y <= 65535, "sg_gemm: m=%d too large for one launch", m);
  // split-K (atomic accumulation) for skinny-output / long-reduction shapes such as dW = X^T dY
  int splits = 1, k_per_split = k > 0 ? k : 1;
  long long tiles = (long long)grid.x * grid.y;
  if (k >= 256 && tiles < ctx->num_sms / 2 && (accumulate || ldc == n)) {
    splits = (int)((2LL * ctx->num_sms + tiles - 1) / tiles);
    int max_splits = k >= 8192 ? k / 512 : k / 64;
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
    k_per_split = ((k + splits - 1) / splits + 15) / 16 * 16;
    splits = (k + k_per_split - 1) / k_per_split;
  }
  if (splits > 1) {      // scratch / ticket budget of the deterministic split combine
    long long fl = (long long)tiles * GT_M * GT_N * (splits + (splits + SG_DET_GROUP - 1) / SG_DET_GROUP);
    long long tk = (long long)tiles * (1 + (splits + SG_DET_GROUP - 1) / SG_DET_GROUP);
    if (fl * (long long)sizeof(float) > (long long)SG_DET_SCRATCH_BYTES || tk > SG_DET_TICKETS) {
      splits = 1;
      k_per_split = k > 0 ? k : 1;
    }
  }
  grid.z = splits;
  // (a one-shot GT_K = 64 instantiation for K <= 64 measured SLOWER than the 16-wide loop on the CBN Dense layers --
  //  19 us vs 10 us per launch in profiles/r01_launches_step.csv -- so the generic loop is used for every shape)
  sg_launch(ctx, k_gemm<16>, grid, 256, 0, trans_a, trans_b, m, n, k, a, lda, b, ldb, c, ldc, bias, accumulate, k_per_split, ctx->det_scratch, ctx->det_tickets);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

// ---------------------------------------------------------------------------------------------------
// Grouped conditional-batch-norm Dense layers (resnet_ops.py:18-26): the generator has 6 CBN layers x (gamma, beta), each a
// bias-free Dense(32 -> C) of the block's 32-wide slice of z.  One launch computes all twelve (forward) and one launch all
// twelve filter gradients (backward) instead of 12 + 12 tiny GEMM launches.
// ---------------------------------------------------------------------------------------------------
#define CBN_MAX_SEG 16
struct CbnSegs {
  int nseg, total;
  int col0[CBN_MAX_SEG], c[CBN_MAX_SEG], z_off[CBN_MAX_SEG];
  long long w_off[CBN_MAX_SEG];
  const float* s[CBN_MAX_SEG];          // backward: upstream [n, c] of the segment
};

// out[r, col] = sum_k z[r, z_off(seg) + k] * W_seg[k, col - col0(seg)],  k < 32
__global__ void __launch_bounds__(256) k_cbn_dense_fwd(const float* __restrict__ z, int z_stride, int n, CbnSegs t,
                                                       const float* __restrict__ w, float* __restrict__ out) {
  const long long total = (long long)n * t.total;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % t.total), r = (int)(i / t.total);
    int sg = 0;
    while (sg + 1 < t.nseg && col >= t.col0[sg + 1]) ++sg;
    const int cl = col - t.col0[sg], c = t.c[sg];
    const float* zz = z + (long long)r * z_stride + t.z_off[sg];
    const float* ww = w + t.w_off[sg] + cl;
    float acc = 0.f;
#pragma unroll 8
    for (int k = 0; k < 32; ++k) acc = fmaf(zz[k], ww[(long long)k * c], acc);
    out[i] = acc;
  }
}
// dW_seg[k, cl] += sum_r z[r, z_off + k] * s_seg[r, cl]     (one thread per output: no atomics, fixed order over r)
__global__ void __launch_bounds__(256) k_cbn_dense_wgrad(const float* __restrict__ z, int z_stride, int n, CbnSegs t,
                                                         float* __restrict__ dw) {
  const long long total = 32LL * t.total;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % t.total), k = (int)(i / t.total);
    int sg = 0;
    while (sg + 1 < t.nseg && col >= t.col0[sg + 1]) ++sg;
    const int cl = col - t.col0[sg], c = t.c[sg];
    const float* ss = t.s[sg] + cl;
    const float* zz = z + t.z_off[sg] + k;
    float acc = 0.f;
#pragma unroll 4
    for (int r = 0; r < n; ++r) acc = fmaf(zz[(long long)r * z_stride], ss[(long long)r * c], acc);
    dw[t.w_off[sg] + (long long)k * c + cl] += acc;
  }
}

static int cbn_fill(CbnSegs* t, int nseg, const int* c, const int* z_off, const long long* w_off, const char* who) {
  SG_REQUIRE(nseg >= 1 && nseg <= CBN_MAX_SEG && c && z_off && w_off, "%s: bad segment table", who);
  t->nseg = nseg;
  int col = 0;
  for (int i = 0; i < nseg; ++i) {
    SG_REQUIRE(c[i] > 0 && z_off[i] >= 0 && w_off[i] >= 0, "%s: bad segment %d", who, i);
    t->col0[i] = col; t->c[i] = c[i]; t->z_off[i] = z_off[i]; t->w_off[i] = w_off[i]; t->s[i] = nullptr;
    col += c[i];
  }
  t->total = col;
  return SG_OK;
}

/* out[n, sum c] = for every segment i: z[:, z_off[i] : z_off[i] + 32] @ W_i, W_i = w_base + w_off[i] of shape (32, c[i]) */
extern "C" int sg_cbn_dense_fwd(sg_ctx* ctx, const float* z, int z_stride, int n, int nseg, const int* c, const int* z_off,
                                const long long* w_off, const float* w_base, float* out) {
  SG_REQUIRE(ctx && z && w_base && out && n >= 0, "sg_cbn_dense_fwd: bad args");
  CbnSegs t;
  int rc = cbn_fill(&t, nseg, c, z_off, w_off, "sg_cbn_dense_fwd");
  if (rc != SG_OK) return rc;
  if (n == 0) return SG_OK;
  long long need = ((long long)n * t.total + 255) / 256, cap = (long long)ctx->num_sms * 8;
  sg_launch(ctx, k_cbn_dense_fwd, (int)(need < cap ? need : cap), 256, 0, z, z_stride, n, t, w_base, out);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

/* dW_i (at dw_base + w_off[i], shape (32, c[i])) += z[:, z_off[i] : +32]^T @ s_i, s_i = upstream[i] of shape (n, c[i]) */
extern "C" int sg_cbn_dense_wgrad(sg_ctx* ctx, const float* z, int z_stride, int n, int nseg, const int* c, const int* z_off,
                                  const long long* w_off, const float* const* upstream, float* dw_base) {
  SG_REQUIRE(ctx && z && upstream && dw_base && n >= 0, "sg_cbn_dense_wgrad: bad args");
  CbnSegs t;
  int rc = cbn_fill(&t, nseg, c, z_off, w_off, "sg_cbn_dense_wgrad");
  if (rc != SG_OK) return rc;
  for (int i = 0; i < nseg; ++i) {
    SG_REQUIRE(upstream[i] != nullptr, "sg_cbn_dense_wgrad: NULL upstream %d", i);
    t.s[i] = upstream[i];
  }
  if (n == 0) return SG_OK;
  long long need = (32LL * t.total + 255) / 256, cap = (long long)ctx->num_sms * 8;
  sg_launch(ctx, k_cbn_dense_wgrad, (int)(need < cap ? need : cap), 256, 0, z, z_stride, n, t, dw_base);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}
