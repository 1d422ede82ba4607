// One-shot SUM all-reduce of SMALL vectors over NVLink peer memory, fused into the kernels that produce / consume them.
//
// The data-parallel train step has two latency-bound exchange points (SURVEY.md section 8e): batch-norm raw sums
// ([2C] floats, 7 layers forward + 7 backward) and the loss / gradient-balance sums (16 doubles).  A NCCL call costs
// 25-40 us each there (launch + stream hand-shakes), ~15 times per step.  Here every rank owns one buffer in
// symmetric memory (torch.distributed._symmetric_memory: same allocation on every GPU, peers mapped into this
// process' address space, full NVLink 5 bandwidth to any peer through NVSwitch):
//     [2 slots][SG_PEER_SLOT_BYTES]  payload, double buffered by the call sequence number
//     [SG_PEER_MAX_WORLD] uint32     flags: flags[r] = last sequence number rank r has published to me
//     uint32                         my call sequence counter (device resident, so that the exchange can sit inside a
//                                    replayed CUDA graph: every launch reads it, uses counter + 1 and stores it back)
// One launch: (1) write my payload into my slot, (2) system-scope release + store my sequence number into every
// peer's flag word (a remote NVLink write), (3) spin until every peer's flag in MY buffer reached the sequence number,
// (4) read all ranks' payloads (remote NVLink reads, .cv so a stale L1 line is never used) and sum them in RANK ORDER,
// so every replica gets bit-identical results.  Double buffering is safe because a rank can only publish call s+1
// after it finished reading in call s, and nobody overwrites slot (s & 1) before call s+2, which needs all flags of s+1.
// A spin that never completes (~1 minute) traps: a protocol bug must fault, not hang the GPU.
//
// k_bn_finalize_peer fuses that exchange between the second stage of the batch-norm statistics reduction and the
// mean / rstd / moving-average finalisation: reduce partials -> exchange -> finalize in ONE launch.
#include "common.cuh"

#define SG_PEER_MAX_WORLD 16
#define SG_PEER_SLOT_BYTES 16384

struct PeerTable {
  unsigned long long buf[SG_PEER_MAX_WORLD];     // peer buffer base addresses, as mapped in this process
  int world, rank;
  unsigned int seq;                              // filled in on the device from the counter in my buffer
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned int* peer_flags(unsigned long long base) {
  return reinterpret_cast<unsigned int*>(base + 2ull * SG_PEER_SLOT_BYTES);
}

__device__ __forceinline__ unsigned int* peer_counter(unsigned long long base) { return peer_flags(base) + SG_PEER_MAX_WORLD; }
// every thread reads the same value: the counter is only written at the very end of the previous launch on this stream
__device__ __forceinline__ unsigned int peer_next_seq(const PeerTable& pt) { return *peer_counter(pt.buf[pt.rank]) + 1u; }
__device__ __forceinline__ void peer_commit_seq(const PeerTable& pt) {
  __syncthreads();
  if (threadIdx.x == 0) *peer_counter(pt.buf[pt.rank]) = pt.seq;
}

// steps (2) and (3); call with ALL threads of the block after the payload stores, returns with the peers' data visible
__device__ __forceinline__ void peer_publish_and_wait(const PeerTable& pt) {
  __threadfence_system();
  __syncthreads();
  const int t = threadIdx.x;
  if (t < pt.world && t != pt.rank) st_release_sys(peer_flags(pt.buf[t]) + pt.rank, pt.seq);
  if (t < pt.world && t != pt.rank) {
    const unsigned int* f = peer_flags(pt.buf[pt.rank]) + t;
    // bounded spin: replicas can be skewed by seconds on their first steps (module loading, graph capture), so the
    // bound is generous (~1 min); a peer that never arrives still faults instead of hanging the GPU forever
    unsigned int spins = 0;
    while ((int)(ld_acquire_sys(f) - pt.seq) < 0) {
      if (++spins > (1u << 28)) __trap();
      __nanosleep(spins < 4096 ? 20 : 200);
    }
  }
  __syncthreads();
}

template <typename T>
__global__ void __launch_bounds__(512) k_peer_allreduce(T* __restrict__ data, int n, PeerTable pt) {
  pt.seq = peer_next_seq(pt);
  const size_t slot = (size_t)(pt.seq & 1u) * SG_PEER_SLOT_BYTES;
  T* mine = reinterpret_cast<T*>(pt.buf[pt.rank] + slot);
  for (int i = threadIdx.x; i < n; i += blockDim.x) mine[i] = data[i];
  peer_publish_and_wait(pt);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    // all remote reads first (independent, in flight together: one NVLink round trip instead of world - 1), then the sum in
    // rank order
    T vals[SG_PEER_MAX_WORLD];
#pragma unroll
    for (int r = 0; r < SG_PEER_MAX_WORLD; ++r)
      if (r < pt.world) vals[r] = __ldcv(reinterpret_cast<const T*>(pt.buf[r] + slot) + i);
    T acc = 0;
#pragma unroll
    for (int r = 0; r < SG_PEER_MAX_WORLD; ++r)
      if (r < pt.world) acc += vals[r];
    data[i] = acc;
  }
  peer_commit_seq(pt);
}

// second stage of the BN statistics (see bn.cu: partial[nblocks][2c]) + exchange + finalize, one block of 1024 threads
__global__ void __launch_bounds__(1024) k_bn_finalize_peer(const float* __restrict__ partial, int nblocks, int c, double count_total,
                                                            float eps, float momentum, float* __restrict__ sums_out,
                                                            float* __restrict__ mean, float* __restrict__ rstd,
                                                            float* __restrict__ mm, float* __restrict__ mv, PeerTable pt) {
  __shared__ double red[1024];
  pt.seq = peer_next_seq(pt);
  const int c2 = 2 * c;
  const size_t slot = (size_t)(pt.seq & 1u) * SG_PEER_SLOT_BYTES;
  float* mine = reinterpret_cast<float*>(pt.buf[pt.rank] + slot);
  // stage 2 of the statistics: 1024 threads = (c2p columns) x (slices of the per-block partials), double accumulation
  int c2p = 32;
  while (c2p < c2 && c2p < 1024) c2p <<= 1;
  const int slices = 1024 / c2p;
  for (int j0 = 0; j0 < c2; j0 += c2p) {
    const int j = j0 + (threadIdx.x % c2p), sl = threadIdx.x / c2p;
    double t = 0.0;
    if (j < c2)
      for (int b = sl; b < nblocks; b += slices) t += (double)partial[(long long)b * c2 + j];
    __syncthreads();
    red[threadIdx.x] = t;
    __syncthreads();
    if (sl == 0 && j < c2) {
      for (int k = 1; k < slices; ++k) t += red[k * c2p + (threadIdx.x % c2p)];
      mine[j] = (float)t;
    }
  }
  if (pt.world > 1) peer_publish_and_wait(pt);
  else __syncthreads();
  for (int j = threadIdx.x; j < c; j += blockDim.x) {
    float v1[SG_PEER_MAX_WORLD], v2[SG_PEER_MAX_WORLD];            // all remote reads in flight together, then the sums in rank order
#pragma unroll
    for (int r = 0; r < SG_PEER_MAX_WORLD; ++r)
      if (r < pt.world) {
        const float* pr = reinterpret_cast<const float*>(pt.buf[r] + slot);
        v1[r] = __ldcv(pr + j);
        v2[r] = __ldcv(pr + c + j);
      }
    double s = 0.0, ss = 0.0;
#pragma unroll
    for (int r = 0; r < SG_PEER_MAX_WORLD; ++r)
      if (r < pt.world) { s += (double)v1[r]; ss += (double)v2[r]; }
    if (sums_out) { sums_out[j] = (float)s; sums_out[c + j] = (float)ss; }
    double m = s / count_total;
    double var = ss / count_total - m * m;
    if (var < 0.0) var = 0.0;
    mean[j] = (float)m;
    rstd[j] = (float)(1.0 / sqrt(var + (double)eps));
    if (mm) mm[j] = mm[j] * momentum + (float)m * (1.f - momentum);
    if (mv) {
      double unb = count_total > 1.0 ? var * (count_total / (count_total - 1.0)) : var;
      mv[j] = mv[j] * momentum + (float)unb * (1.f - momentum);
    }
  }
  peer_commit_seq(pt);
}

// barrier only: publish my next sequence number to every peer, wait for theirs
__global__ void __launch_bounds__(32) k_peer_barrier(PeerTable pt) {
  pt.seq = peer_next_seq(pt);
  peer_publish_and_wait(pt);
  peer_commit_seq(pt);
}

// my shard of the gradient bucket: g[i] = sum over ranks, in RANK order, of that rank's copy (mine in place, the peers' from the
// staging slots the copy engines filled): the same additions in the same order whichever rank owns the shard
__global__ void __launch_bounds__(256) k_bucket_reduce(float* __restrict__ g, const float* __restrict__ staging, long long len,
                                                        long long slot_stride, int world, int rank) {
  const long long n4 = len / 4, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int slot = 0;
    for (int r = 0; r < world; ++r) {
      float4 v = (r == rank) ? sg_ld4(g + 4 * i) : sg_ld4(staging + (long long)(slot++) * slot_stride + 4 * i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    sg_st4(g + 4 * i, acc);
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) {
    float acc = 0.f;
    int slot = 0;
    for (int r = 0; r < world; ++r) acc += (r == rank) ? g[i] : staging[(long long)(slot++) * slot_stride + i];
    g[i] = acc;
  }
}

// The same reduce-scatter / all-gather with the SMs doing the NVLink reads (for a bucket whose all-reduce is EXPOSED -- nothing
// else left to run beside it -- the whole machine pulling over NVLink beats one copy engine per peer).
struct BucketPtrs { unsigned long long g[SG_PEER_MAX_WORLD]; };

__global__ void __launch_bounds__(256) k_bucket_pull_reduce(BucketPtrs bp, long long lo, long long len, int world, int rank) {
  float* mine = reinterpret_cast<float*>(bp.g[rank]) + lo;
  const long long n4 = len / 4, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    // every replica's copy first (independent NVLink reads in flight together), then the sum in rank order: the same
    // additions whichever replica owns the shard
    float4 v[SG_PEER_MAX_WORLD];
#pragma unroll
    for (int r = 0; r < SG_PEER_MAX_WORLD; ++r)
      if (r < world) v[r] = __ldcg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(bp.g[r]) + lo) + i);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < SG_PEER_MAX_WORLD; ++r)
      if (r < world) { acc.x += v[r].x; acc.y += v[r].y; acc.z += v[r].z; acc.w += v[r].w; }
    __stcg(reinterpret_cast<float4*>(mine) + i, acc);
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) {
    float acc = 0.f;
    for (int r = 0; r < world; ++r) acc += __ldcg(reinterpret_cast<const float*>(bp.g[r]) + lo + i);
    mine[i] = acc;
  }
}

// all-gather: blockIdx.y = peer index (skipping myself); copy that peer's reduced shard into my bucket
__global__ void __launch_bounds__(256) k_bucket_gather(BucketPtrs bp, long long shard, long long n, int world, int rank) {
  const int r = (int)blockIdx.y < rank ? (int)blockIdx.y : (int)blockIdx.y + 1;
  long long lo = (long long)r * shard, hi = lo + shard;
  if (lo > n) lo = n;
  if (hi > n) hi = n;
  const long long len = hi - lo;
  const float* src = reinterpret_cast<const float*>(bp.g[r]) + lo;
  float* dst = reinterpret_cast<float*>(bp.g[rank]) + lo;
  const long long n4 = len / 4, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride)
    __stcg(reinterpret_cast<float4*>(dst) + i, __ldcg(reinterpret_cast<const float4*>(src) + i));
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) dst[i] = __ldcg(src + i);
}

static int make_table(PeerTable* pt, const unsigned long long* peer_bufs, int world, int rank, const char* who) {
  SG_REQUIRE(peer_bufs && world >= 1 && world <= SG_PEER_MAX_WORLD && rank >= 0 && rank < world, "%s: bad peer table", who);
  memset(pt, 0, sizeof(*pt));
  for (int r = 0; r < world; ++r) {
    SG_REQUIRE(peer_bufs[r] != 0 && (peer_bufs[r] & 15) == 0, "%s: peer buffer %d is NULL or misaligned", who, r);
    pt->buf[r] = peer_bufs[r];
  }
  pt->world = world; pt->rank = rank; pt->seq = 0;
  return SG_OK;
}

extern "C" {

size_t sg_peer_buffer_bytes(void) { return 2 * (size_t)SG_PEER_SLOT_BYTES + (SG_PEER_MAX_WORLD + 1) * sizeof(unsigned int) + 60; }
size_t sg_peer_max_payload_bytes(void) { return SG_PEER_SLOT_BYTES; }

int sg_peer_allreduce_sum(sg_ctx* ctx, void* data, int n, int is_f64, const unsigned long long* peer_bufs, int world, int rank) {
  SG_REQUIRE(ctx && data && n >= 0, "sg_peer_allreduce_sum: bad args");
  SG_REQUIRE((size_t)n * (is_f64 ? 8 : 4) <= SG_PEER_SLOT_BYTES, "sg_peer_allreduce_sum: payload of %d elements exceeds the slot", n);
  if (n == 0 || world <= 1) return SG_OK;
  PeerTable pt;
  int rc = make_table(&pt, peer_bufs, world, rank, "sg_peer_allreduce_sum");
  if (rc != SG_OK) return rc;
  int threads = n >= 512 ? 512 : (n >= 256 ? 256 : 128);
  if (threads < 32 * ((world + 31) / 32)) threads = 32 * ((world + 31) / 32);
  if (is_f64) sg_launch(ctx, k_peer_allreduce<double>, 1, threads, 0, (double*)data, n, pt);
  else sg_launch(ctx, k_peer_allreduce<float>, 1, threads, 0, (float*)data, n, pt);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

int sg_peer_barrier(sg_ctx* ctx, const unsigned long long* peer_bufs, int world, int rank) {
  SG_REQUIRE(ctx != nullptr, "sg_peer_barrier: ctx is NULL");
  if (world <= 1) return SG_OK;
  PeerTable pt;
  int rc = make_table(&pt, peer_bufs, world, rank, "sg_peer_barrier");
  if (rc != SG_OK) return rc;
  sg_launch(ctx, k_peer_barrier, 1, 32, 0, pt);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

static int bucket_aux_streams(sg_ctx* ctx, int want) {
  if (want > 8) want = 8;
  if (want < 1) want = 1;
  while (ctx->n_aux < want) {
    if (ctx->n_aux == 0) SG_CHECK_CUDA(cudaEventCreateWithFlags(&ctx->aux_fork, cudaEventDisableTiming));
    SG_CHECK_CUDA(cudaStreamCreateWithFlags(&ctx->aux_stream[ctx->n_aux], cudaStreamNonBlocking));
    SG_CHECK_CUDA(cudaEventCreateWithFlags(&ctx->aux_join[ctx->n_aux], cudaEventDisableTiming));
    ++ctx->n_aux;
  }
  return SG_OK;
}

long long sg_peer_bucket_shard(long long n, int world) {
  long long s = (n + world - 1) / world;
  return (s + 3) / 4 * 4;                 // 16-byte aligned shard starts
}

int sg_peer_bucket_allreduce(sg_ctx* ctx, float* g, long long n, float* staging, const unsigned long long* g_ptrs,
                             const unsigned long long* flag_bufs, int world, int rank, int use_sms) {
  SG_REQUIRE(ctx && g && n >= 0 && world >= 1 && world <= SG_PEER_MAX_WORLD && rank >= 0 && rank < world, "sg_peer_bucket_allreduce: bad args");
  if (world == 1 || n == 0) return SG_OK;
  SG_REQUIRE(staging && g_ptrs && flag_bufs && (float*)(uintptr_t)g_ptrs[rank] == g && ((uintptr_t)g & 15) == 0 && ((uintptr_t)staging & 15) == 0,
             "sg_peer_bucket_allreduce: needs a staging buffer, the peer table of the bucket (g_ptrs[rank] == g) and 16-byte alignment");
  const long long shard = sg_peer_bucket_shard(n, world);
  auto lo = [&](int r) { long long a = (long long)r * shard; return a < n ? a : n; };
  auto len = [&](int r) { return lo(r + 1) - lo(r); };
  // (1) every replica's bucket is complete (stream order on each rank + barrier)
  int rc = sg_peer_barrier(ctx, flag_bufs, world, rank);
  if (rc != SG_OK) return rc;
  if (use_sms) {
    BucketPtrs bp;
    memset(&bp, 0, sizeof(bp));
    for (int r = 0; r < world; ++r) bp.g[r] = g_ptrs[r];
    const long long mylen_ = len(rank);
    if (mylen_ > 0) {
      long long need = (mylen_ / 4 + 255) / 256, cap = (long long)ctx->num_sms * 4;
      sg_launch(ctx, k_bucket_pull_reduce, (int)(need < cap ? (need < 1 ? 1 : need) : cap), 256, 0, bp, lo(rank), mylen_, world, rank);
      SG_POST_LAUNCH(ctx);
    }
    rc = sg_peer_barrier(ctx, flag_bufs, world, rank);
    if (rc != SG_OK) return rc;
    {
      long long need = (shard / 4 + 255) / 256, cap = (long long)ctx->num_sms * 4 / (world - 1) + 1;
      dim3 grid((unsigned)(need < cap ? (need < 1 ? 1 : need) : cap), (unsigned)(world - 1));
      sg_launch(ctx, k_bucket_gather, grid, 256, 0, bp, shard, n, world, rank);
      SG_POST_LAUNCH(ctx);
    }
    return sg_peer_barrier(ctx, flag_bufs, world, rank);
  }
  // (2) reduce-scatter, pull side: the copy engines fetch MY shard of every peer's bucket over NVLink (no SM involved), one
  //     pull per auxiliary stream so that the pulls from different peers run concurrently (fork / join by events: capturable)
  rc = bucket_aux_streams(ctx, world - 1);
  if (rc != SG_OK) return rc;
  const long long mylen = len(rank);
  if (mylen > 0) {
    SG_CHECK_CUDA(cudaEventRecord(ctx->aux_fork, ctx->stream));
    int slot = 0;
    for (int r = 0; r < world; ++r) {
      if (r == rank) continue;
      cudaStream_t st = ctx->aux_stream[slot % ctx->n_aux];
      if (slot < ctx->n_aux) SG_CHECK_CUDA(cudaStreamWaitEvent(st, ctx->aux_fork, 0));
      SG_CHECK_CUDA(cudaMemcpyAsync(staging + (long long)slot * shard, (const float*)(uintptr_t)g_ptrs[r] + lo(rank), (size_t)mylen * sizeof(float),
                                    cudaMemcpyDeviceToDevice, st));
      ++slot;
    }
    for (int k = 0; k < ctx->n_aux && k < world - 1; ++k) {
      SG_CHECK_CUDA(cudaEventRecord(ctx->aux_join[k], ctx->aux_stream[k]));
      SG_CHECK_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->aux_join[k], 0));
    }
    long long need = (mylen / 4 + 255) / 256;
    int grid = (int)(need < 64 ? (need < 1 ? 1 : need) : 64);       // a small grid: this runs under the step's compute kernels
    sg_launch(ctx, k_bucket_reduce, grid, 256, 0, g + lo(rank), staging, mylen, shard, world, rank);
    SG_POST_LAUNCH(ctx);
  }
  // (3) every shard is reduced on its owner
  rc = sg_peer_barrier(ctx, flag_bufs, world, rank);
  if (rc != SG_OK) return rc;
  // (4) all-gather, pull side, again one peer per auxiliary stream
  {
    SG_CHECK_CUDA(cudaEventRecord(ctx->aux_fork, ctx->stream));
    int slot = 0;
    for (int r = 0; r < world; ++r) {
      if (r == rank) continue;
      cudaStream_t st = ctx->aux_stream[slot % ctx->n_aux];
      if (slot < ctx->n_aux) SG_CHECK_CUDA(cudaStreamWaitEvent(st, ctx->aux_fork, 0));
      if (len(r) > 0)
        SG_CHECK_CUDA(cudaMemcpyAsync(g + lo(r), (const float*)(uintptr_t)g_ptrs[r] + lo(r), (size_t)len(r) * sizeof(float), cudaMemcpyDeviceToDevice, st));
      ++slot;
    }
    for (int k = 0; k < ctx->n_aux && k < world - 1; ++k) {
      SG_CHECK_CUDA(cudaEventRecord(ctx->aux_join[k], ctx->aux_stream[k]));
      SG_CHECK_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->aux_join[k], 0));
    }
  }
  // (5) nobody touches its bucket again before every peer has read its shard
  return sg_peer_barrier(ctx, flag_bufs, world, rank);
}

/* BN statistics, stage 2 + cross-replica exchange + finalize (replaces k_bn_stats_reduce, the NCCL all-reduce and
 * k_bn_finalize).  `partial` / `nblocks` come from sg_bn_stats_partial.  count_total = rows summed over all replicas. */
int sg_bn_finalize_peer(sg_ctx* ctx, const float* partial, int nblocks, int c, double count_total, float eps, float momentum,
                        float* sums_out, float* mean, float* rstd, float* moving_mean, float* moving_var,
                        const unsigned long long* peer_bufs, int world, int rank) {
  SG_REQUIRE(ctx && partial && mean && rstd && nblocks >= 1 && c > 0, "sg_bn_finalize_peer: bad args");
  SG_REQUIRE((size_t)c * 8 <= SG_PEER_SLOT_BYTES, "sg_bn_finalize_peer: c=%d exceeds the slot", c);
  PeerTable pt;
  int rc = make_table(&pt, peer_bufs, world, rank, "sg_bn_finalize_peer");
  if (rc != SG_OK) return rc;
  sg_launch(ctx, k_bn_finalize_peer, 1, 1024, 0, partial, nblocks, c, count_total, eps, momentum, sums_out, mean, rstd, moving_mean,
                                                 moving_var, pt);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

}  // extern "C"
