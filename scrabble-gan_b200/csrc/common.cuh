// Shared device/host helpers for libsgan (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/sgan.h"

struct sg_ctx {
  int device;
  cudaStream_t stream;
  int num_sms;
  void* encode_tiled;        // PFN cuTensorMapEncodeTiled (resolved lazily)
  long long launches;        // number of kernels launched through this context
  int speed_mode;            // 1: bf16 speed mode -- small fp32 GEMMs of the non-local block use bf16 warp-level tensor ops
  // fixed workspace of the deterministic cross-block reductions (allocated once by sg_ctx_create, see sg_det_* below):
  float* det_scratch;        // SG_DET_SCRATCH_BYTES of per-block partial sums
  unsigned int* det_tickets; // SG_DET_TICKETS arrival counters / turn semaphores, all zero between launches
  int conv_split_tail;       // k_conv_tc: split the k-range of the tiles of a partial last wave (sg_ctx_set_conv_split_tail)
  // auxiliary streams of the copy-engine gradient-bucket all-reduce (peer.cu): one peer pull per stream, so that the pulls
  // from different peers run on different copy engines at the same time; created on first use
  cudaStream_t aux_stream[8];
  cudaEvent_t aux_fork, aux_join[8];
  int n_aux;
};
#define SG_DET_SCRATCH_BYTES (48u << 20)
#define SG_DET_TICKETS 16384

void sg_set_error(const char* fmt, ...);

#define SG_CHECK_CUDA(expr)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      sg_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__,    \
                   cudaGetErrorString(_e));                                                   \
      return SG_ERR_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

#define SG_REQUIRE(cond, ...)                                                                 \
  do {                                                                                        \
    if (!(cond)) {                                                                            \
      sg_set_error(__VA_ARGS__);                                                              \
      return SG_ERR_ARG;                                                                      \
    }                                                                                         \
  } while (0)

#define SG_POST_LAUNCH(ctx)                                                                   \
  do {                                                                                        \
    (ctx)->launches++;                                                                        \
    SG_CHECK_CUDA(cudaGetLastError());                                                        \
  } while (0)

static inline int sg_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------------------
// Kernel launches
// ---------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
template <typename... P, typename... A>
static inline cudaError_t sg_launch_ex(sg_ctx* ctx, bool cooperative, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, A&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  memset(attr, 0, sizeof(attr));
  attr[0].id = cudaLaunchAttributeCooperative;   // grid-wide barrier inside: the runtime guarantees (or refuses) co-residency
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cooperative ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<P>(args)...);
}
// errors surface through the SG_POST_LAUNCH that follows every launch (cudaGetLastError)
template <typename... P, typename... A>
static inline void sg_launch(sg_ctx* ctx, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, A&&... args) {
  (void)sg_launch_ex(ctx, false, kern, grid, block, smem, args...);
}
#endif

// ---------------------------------------------------------------------------------------------------
// typed load / store helpers (operand tensors are fp32 or bf16; arithmetic is always fp32)
// ---------------------------------------------------------------------------------------------------
template <typename T> struct sg_dt;
template <> struct sg_dt<float> { static constexpr int id = SG_F32; };
template <> struct sg_dt<__nv_bfloat16> { static constexpr int id = SG_BF16; };

__device__ __forceinline__ float sg_ld(const float* p) { return *p; }
__device__ __forceinline__ float sg_ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void sg_st(float* p, float v) { *p = v; }
__device__ __forceinline__ void sg_st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

__device__ __forceinline__ float4 sg_ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 sg_ld4(const __nv_bfloat16* p) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&r.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&r.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void sg_st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void sg_st4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&a);
  r.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = r;
}

__device__ __forceinline__ float sg_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float sg_warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum (blockDim.x multiple of 32, <= 1024); result valid in all threads
__device__ __forceinline__ float sg_block_sum(float v, float* smem32) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = sg_warp_sum(v);
  __syncthreads();
  if (lane == 0) smem32[w] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  float r = (threadIdx.x < nw) ? smem32[threadIdx.x] : 0.f;
  if (w == 0) {
    r = sg_warp_sum(r);
    if (lane == 0) smem32[0] = r;
  }
  __syncthreads();
  return smem32[0];
}

// ---------------------------------------------------------------------------------------------------
// Deterministic cross-block reductions.  Floating-point atomics make a sum depend on the arrival order of the blocks;
// the two schemes below fix the order, so that gradients are bitwise repeatable from run to run.
//   (B) partials + last block: every block of a group stores its partial vector in its own scratch slot, takes a ticket,
//       and the block that arrives LAST sums the slots in block-index order (whichever block that is, the order of the
//       additions is the same).  Used where the output is small and many blocks contribute (bias / BN sums, dot, ...).
//   (A) ordered turns: split s of an output tile waits until splits 0..s-1 have added their partial tiles (a semaphore per
//       tile), then adds its own.  A waiting block only ever waits on blocks with a LOWER linear block index (dispatched
//       before it; in the persistent tensor-core kernel: on units processed earlier), so the wait always ends.  Used for
//       the filter-gradient kernels (large output tiles, few splits).
// Tickets / semaphores are left at zero by the last arrival, so launches on one stream can share them.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool sg_det_arrive_last(unsigned int* ticket, unsigned int nblk) {
  __shared__ unsigned int s_last;
  __threadfence();                    // this block's partials are visible device-wide before its ticket
  __syncthreads();
  if (threadIdx.x == 0 && threadIdx.y == 0 && threadIdx.z == 0) {
    unsigned int t = atomicAdd(ticket, 1u);
    s_last = (t == nblk - 1) ? 1u : 0u;
    if (s_last) *ticket = 0u;
  }
  __syncthreads();
  const bool last = s_last != 0u;
  if (last) __threadfence();
  return last;
}
// sum over slots [b0, b1) (slot stride `n` floats) of element j, in a FIXED association (eight interleaved chains, so that
// the L2 loads -- the slots were written by other SMs -- overlap instead of forming one long dependent chain)
__device__ __forceinline__ float sg_det_range_sum(const float* slots, unsigned int b0, unsigned int b1, long long n, long long j) {
  float a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = 0.f;
  unsigned int b = b0;
  for (; b + 7 < b1; b += 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] += __ldcg(slots + (long long)(b + k) * n + j);
  }
  for (; b < b1; ++b) a[0] += __ldcg(slots + (long long)b * n + j);
  return ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
}
// Block-cooperative ordered sum of `nblk` slots of `n` floats (1-D blocks of <= 1024 threads; ALL threads must call).  When
// the block has more threads than elements, the slots are cut into up to 32 contiguous ranges summed by different threads and
// combined in range order through shared memory.  emit(j, total) runs once per element.  The result depends only on
// (nblk, n, blockDim), never on timing.
template <class Emit>
__device__ __forceinline__ void sg_det_block_reduce(const float* slots, unsigned int nblk, int n, Emit emit) {
  __shared__ float part_sm[1024];
  const int nt = blockDim.x, tid = threadIdx.x;
  if (n >= nt) {
    // at least one element per thread: every thread walks the slots in order for FOUR of its elements at a time, so that
    // four (x2 by unrolling) independent L2 loads are in flight instead of one dependent chain
    for (int j0 = tid; j0 < n; j0 += 4 * nt) {
      const int j1 = j0 + nt, j2 = j0 + 2 * nt, j3 = j0 + 3 * nt;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 2
      for (unsigned int b = 0; b < nblk; ++b) {
        const float* row = slots + (long long)b * n;
        a0 += __ldcg(row + j0);
        if (j1 < n) a1 += __ldcg(row + j1);
        if (j2 < n) a2 += __ldcg(row + j2);
        if (j3 < n) a3 += __ldcg(row + j3);
      }
      emit(j0, a0);
      if (j1 < n) emit(j1, a1);
      if (j2 < n) emit(j2, a2);
      if (j3 < n) emit(j3, a3);
    }
    return;
  }
  // fewer elements than threads: the slots are cut into up to 32 contiguous ranges summed by different threads and
  // combined in range order through shared memory
  int P = nt / n;
  if (P > 32) P = 32;
  if (P > (int)nblk) P = (int)nblk;
  const int jl = tid % n, part = tid / n;
  if (part < P) {
    const unsigned int chunk = (nblk + P - 1) / P;
    unsigned int b0 = part * chunk, b1 = b0 + chunk;
    if (b1 > nblk) b1 = nblk;
    part_sm[part * n + jl] = b0 < b1 ? sg_det_range_sum(slots, b0, b1, n, jl) : 0.f;
  }
  __syncthreads();
  if (part == 0) {
    float t = 0.f;
    for (int q = 0; q < P; ++q) t += part_sm[q * n + jl];
    emit(jl, t);
  }
  __syncthreads();
}
// Scheme (B) in full: block `bi` of `nblk` has stored its partial vector in slots[bi * n ...].  Up to 32 blocks: the last
// arrival sums all slots.  More: two levels -- the last arrival of each group of 16 consecutive blocks sums its group into
// slots2[group * n ...], and the last group to finish sums the groups -- so no thread ever walks more than ~40 slots.
// tickets: 1 + ceil(nblk / 16) counters (zero between launches); slots2: ceil(nblk / 16) * n floats.
#define SG_DET_GROUP 16
template <class Emit>
__device__ __forceinline__ void sg_det_finish(const float* slots, float* slots2, unsigned int* tickets, unsigned int nblk, unsigned int bi, int n,
                                              Emit emit) {
  if (nblk <= 32) {
    if (sg_det_arrive_last(tickets, nblk)) sg_det_block_reduce(slots, nblk, n, emit);
    return;
  }
  const unsigned int ngroups = (nblk + SG_DET_GROUP - 1) / SG_DET_GROUP, grp = bi / SG_DET_GROUP;
  const unsigned int gsize = (grp + 1) * SG_DET_GROUP <= nblk ? SG_DET_GROUP : nblk - grp * SG_DET_GROUP;
  if (!sg_det_arrive_last(tickets + 1 + grp, gsize)) return;
  float* mine = slots2 + (long long)grp * n;
  sg_det_block_reduce(slots + (long long)grp * SG_DET_GROUP * n, gsize, n, [&](int j, float t) { mine[j] = t; });
  if (!sg_det_arrive_last(tickets, ngroups)) return;
  sg_det_block_reduce(slots2, ngroups, n, emit);
}
// floats of scratch one such reduction needs
static inline long long sg_det_floats(long long nblk, long long n) {
  return nblk * n + (nblk > 32 ? (nblk + SG_DET_GROUP - 1) / SG_DET_GROUP * n : 0);
}
__device__ __forceinline__ void sg_turn_wait(unsigned int* sem, unsigned int turn) {
  if (turn == 0) return;
  unsigned int v, spins = 0;
  do {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(sem) : "memory");
    if (v == turn) break;
    if (++spins > (1u << 26)) __trap();      // a protocol bug must fault, never hang the GPU
    __nanosleep(64);
  } while (true);
}
__device__ __forceinline__ void sg_turn_pass(unsigned int* sem, unsigned int turn, unsigned int nturns) {
  unsigned int next = (turn + 1 == nturns) ? 0u : turn + 1;      // the last turn leaves the semaphore at zero
  __threadfence();
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(sem), "r"(next) : "memory");
}

#define SG_DISPATCH_DT(dt, T, ...)                              \
  do {                                                          \
    if ((dt) == SG_F32) {                                       \
      using T = float;                                          \
      __VA_ARGS__;                                              \
    } else if ((dt) == SG_BF16) {                               \
      using T = __nv_bfloat16;                                  \
      __VA_ARGS__;                                              \
    } else {                                                    \
      sg_set_error("bad dtype %d", (int)(dt));                  \
      return SG_ERR_ARG;                                        \
    }                                                           \
  } while (0)
