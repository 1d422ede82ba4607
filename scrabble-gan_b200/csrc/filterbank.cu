// Per-character filter bank (K13).  Reference: arch_ops.py:84-90 (SpatialEmbedding = embedding_lookup) and
// net_architecture.py:260-271 (z0 (1x32) @ bank[y] (32x8192), reshape, reshape, transpose).
// The reference materialises (B,L,32,8192); here each bank element is read straight from bank[vocab,32,8192]
// (54.5 MB, L2-resident across the batch) and written directly in NHWC (B,4,4L,512):
//     out[b, k%4, 4*l + k/2048, (k%2048)/4] = sum_j z0[b,j] * bank[y[b,l], j, k]        (integer map, bit-exact)
#include "common.cuh"

#define FB_J 32
#define FB_K 8192

__device__ __forceinline__ long long fb_out_index(int b, int l, int L, int k) {
  int h = k & 3, w = 4 * l + (k >> 11), c = (k & 2047) >> 2;
  return (((long long)b * 4 + h) * (4 * L) + w) * 512 + c;
}

// grid: (FB_K/256, B*L), block 256: thread = one k
__global__ void __launch_bounds__(256) k_fb_fwd(const float* __restrict__ z, int z_stride, const int* __restrict__ y,
                                                 int L, int vocab, const float* __restrict__ bank,
                                                 float* __restrict__ out) {
  __shared__ float zs[FB_J];
  int p = blockIdx.y, b = p / L, l = p % L;
  int v = y[p];
  if (threadIdx.x < FB_J) zs[threadIdx.x] = z[(long long)b * z_stride + threadIdx.x];
  __syncthreads();
  int k = blockIdx.x * 256 + threadIdx.x;
  float acc = 0.f;
  if (v >= 0 && v < vocab) {
    const float* bp = bank + (long long)v * FB_J * FB_K + k;
#pragma unroll 8
    for (int j = 0; j < FB_J; ++j) acc = fmaf(zs[j], bp[(long long)j * FB_K], acc);
  }
  out[fb_out_index(b, l, L, k)] = acc;
}

// dbank[v, j, k] = sum_{p : y[p]==v} z0[b_p, j] * dout_p[k].   grid: (FB_K/128, vocab), block 128: thread = one k,
// 32 accumulators (one per j).  Deterministic (no atomics); every element of dbank is written.
__global__ void __launch_bounds__(128) k_fb_bwd_bank(const float* __restrict__ dout, const float* __restrict__ z,
                                                      int z_stride, const int* __restrict__ y, int B, int L,
                                                      float* __restrict__ dbank) {
  __shared__ float zs[FB_J];
  int v = blockIdx.y;
  int k = blockIdx.x * 128 + threadIdx.x;
  float acc[FB_J];
#pragma unroll
  for (int j = 0; j < FB_J; ++j) acc[j] = 0.f;
  int P = B * L;
  for (int p = 0; p < P; ++p) {
    if (y[p] != v) continue;          // block-uniform branch
    int b = p / L, l = p % L;
    __syncthreads();
    if (threadIdx.x < FB_J) zs[threadIdx.x] = z[(long long)b * z_stride + threadIdx.x];
    __syncthreads();
    float d = dout[fb_out_index(b, l, L, k)];
#pragma unroll
    for (int j = 0; j < FB_J; ++j) acc[j] = fmaf(zs[j], d, acc[j]);
  }
  float* dp = dbank + (long long)v * FB_J * FB_K + k;
#pragma unroll
  for (int j = 0; j < FB_J; ++j) dp[(long long)j * FB_K] = acc[j];
}

// dz0[b, j] = sum_l sum_k bank[y[b,l], j, k] * dout[b,l,k].   grid: (FB_J, B), block 256
__global__ void __launch_bounds__(256) k_fb_bwd_z(const float* __restrict__ dout, const int* __restrict__ y, int L,
                                                   int vocab, const float* __restrict__ bank, float* __restrict__ dz0,
                                                   int dz_stride) {
  __shared__ float sm[32];
  int j = blockIdx.x, b = blockIdx.y;
  float acc = 0.f;
  for (int l = 0; l < L; ++l) {
    int v = y[b * L + l];
    if (v < 0 || v >= vocab) continue;
    const float* bp = bank + ((long long)v * FB_J + j) * FB_K;
    for (int k = threadIdx.x; k < FB_K; k += 256) acc = fmaf(bp[k], dout[fb_out_index(b, l, L, k)], acc);
  }
  float t = sg_block_sum(acc, sm);
  if (threadIdx.x == 0) dz0[(long long)b * dz_stride + j] = t;
}

extern "C" {

int sg_filterbank_fwd(sg_ctx* ctx, const float* z, int z_stride, const int* y, int b, int l, int vocab,
                      const float* bank, float* out) {
  SG_REQUIRE(ctx && z && y && bank && out, "sg_filterbank_fwd: NULL");
  SG_REQUIRE(b >= 0 && l >= 0 && vocab > 0 && z_stride >= FB_J, "sg_filterbank_fwd: bad sizes");
  if (b * l == 0) return SG_OK;
  dim3 grid(FB_K / 256, b * l);
  sg_launch(ctx, k_fb_fwd, grid, 256, 0, z, z_stride, y, l, vocab, bank, out);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_filterbank_bwd(sg_ctx* ctx, const float* dout, const float* z, int z_stride, const int* y, int b, int l,
                      int vocab, const float* bank, float* dbank, float* dz0, int dz_stride) {
  SG_REQUIRE(ctx && dout && z && y && bank && dbank, "sg_filterbank_bwd: NULL");
  SG_REQUIRE(b >= 0 && l >= 0 && vocab > 0 && z_stride >= FB_J, "sg_filterbank_bwd: bad sizes");
  dim3 grid(FB_K / 128, vocab);
  sg_launch(ctx, k_fb_bwd_bank, grid, 128, 0, dout, z, z_stride, y, b, l, dbank);
  SG_POST_LAUNCH(ctx);
  if (dz0 && b * l > 0) {
    dim3 g2(FB_J, b);
    sg_launch(ctx, k_fb_bwd_z, g2, 256, 0, dout, y, l, vocab, bank, dz0, dz_stride);
    SG_POST_LAUNCH(ctx);
  }
  return SG_OK;
}

}  // extern "C"
