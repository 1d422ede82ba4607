// Fused softmax -> log(p + 1e-7) -> CTC loss -> gradient w.r.t. the Dense pre-activations (K15).
// Reference: net_architecture.py:55 (Dense softmax) and :57-72 (K.ctc_batch_cost):
//     y_pred = log(softmax(z) + 1e-7);  loss = tf.nn.ctc_loss(inputs=y_pred, ...)   (which re-softmaxes its inputs)
// => effective per-frame distribution q = (p + eps) / (1 + C eps), blank = C-1, repeats merged.
// One CTA per sample; thread s owns extended-label state s (S = 2L+1); log-space alpha/beta in shared memory.
// dL/du (u = log(p+eps)) = q - occupancy/P  [tf.nn.ctc_loss gradient], chained through log and softmax to z.
#include <atomic>

#include "common.cuh"

#define CTC_EPS 1e-7f
#define NEG_INF (-INFINITY)

// accurate (not fast-intrinsic) log-sum-exp: the recursion runs T steps in the log domain and its output is
// differenced against log q when forming posteriors, so absolute log-domain error matters (CTC parity 1e-4)
__device__ __forceinline__ float lse2(float a, float b) {
  float m = fmaxf(a, b);
  if (m == NEG_INF) return NEG_INF;
  return m + log1pf(expf(fminf(a, b) - m));
}
__device__ __forceinline__ float lse3(float a, float b, float c) {
  float m = fmaxf(fmaxf(a, b), c);
  if (m == NEG_INF) return NEG_INF;
  // sum of the two non-max terms, then log1p
  float s = expf(a - m) + expf(b - m) + expf(c - m) - 1.f;
  return m + log1pf(s);
}

// frame count of sample b: input_len[b] (all Tmax frames without input_len) clamped to [lo, Tmax]
static __device__ __forceinline__ int sample_frames(const int* input_len, int b, int lo, int Tmax) {
  const int T = input_len ? input_len[b] : Tmax;
  return T < lo ? lo : (T > Tmax ? Tmax : T);
}

// softmax of one row z[0, C), one warp: max-subtracted exp and an fp32 sum; store(k, p_k) for every class
template <class Store>
static __device__ __forceinline__ void warp_softmax_row(const float* z, int C, int lane, Store store) {
  float mx = NEG_INF;
  for (int k = lane; k < C; k += 32) mx = fmaxf(mx, z[k]);
  mx = sg_warp_max(mx);
  float sum = 0.f;
  for (int k = lane; k < C; k += 32) sum += expf(z[k] - mx);
  sum = sg_warp_sum(sum);
  const float inv = 1.f / sum;
  for (int k = lane; k < C; k += 32) store(k, expf(z[k] - mx) * inv);
}

// dynamic smem: logq[T*C] | alpha[T*S] | beta[T*S] | occ[C] | ext[S] (int)
// Ragged batches (K.ctc_batch_cost's own interface: per-sample input_length / label_length, net_architecture.py:57-72):
// input_len / label_len, when given, hold every sample's frame count T_b <= Tmax and label count L_b <= Lmax; logits / labels
// / grad keep the rectangular [b, Tmax, C] / [b, Lmax] layout, frames t >= T_b get a zero gradient.
__global__ void k_ctc(const float* __restrict__ logits, const int* __restrict__ labels, int Tmax, int C, int Lmax,
                      const int* __restrict__ input_len, const int* __restrict__ label_len, float* __restrict__ loss,
                      float* __restrict__ grad) {
  extern __shared__ float sm[];
  const int b = blockIdx.x;
  const int T = sample_frames(input_len, b, 1, Tmax);
  int L = label_len ? label_len[b] : Lmax;
  L = L < 0 ? 0 : (L > Lmax ? Lmax : L);
  const int S = 2 * L + 1, Smax = 2 * Lmax + 1;
  float* logq = sm;
  float* alpha = logq + Tmax * C;
  float* beta = alpha + Tmax * Smax;
  float* occ = beta + Tmax * Smax;
  int* ext = reinterpret_cast<int*>(occ + C);
  __shared__ float s_logp;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int blank = C - 1;
  const float* z = logits + (long long)b * Tmax * C;

  for (int s = tid; s < S; s += blockDim.x) ext[s] = (s & 1) ? labels[b * Lmax + (s >> 1)] : blank;

  // per-frame effective log-probabilities: one warp per frame
  const float log_norm = logf(1.f + (float)C * CTC_EPS);
  for (int t = warp; t < T; t += nwarps)
    warp_softmax_row(z + t * C, C, lane, [&](int k, float p) { logq[t * C + k] = logf(p + CTC_EPS) - log_norm; });
  __syncthreads();

  // alpha recursion
  for (int s = tid; s < S; s += blockDim.x)
    alpha[s] = (s < 2) ? logq[ext[s]] : NEG_INF;
  __syncthreads();
  for (int t = 1; t < T; ++t) {
    for (int s = tid; s < S; s += blockDim.x) {
      const float* prev = alpha + (t - 1) * S;
      float a0 = prev[s];
      float a1 = s >= 1 ? prev[s - 1] : NEG_INF;
      float a2 = (s >= 2 && ext[s] != blank && ext[s] != ext[s - 2]) ? prev[s - 2] : NEG_INF;
      float v = lse3(a0, a1, a2);
      alpha[t * S + s] = (v == NEG_INF) ? NEG_INF : v + logq[t * C + ext[s]];
    }
    __syncthreads();
  }
  // beta recursion (beta_t(s) includes the emission at t)
  for (int s = tid; s < S; s += blockDim.x)
    beta[(T - 1) * S + s] = (s >= S - 2) ? logq[(T - 1) * C + ext[s]] : NEG_INF;
  __syncthreads();
  for (int t = T - 2; t >= 0; --t) {
    for (int s = tid; s < S; s += blockDim.x) {
      const float* nxt = beta + (t + 1) * S;
      float b0 = nxt[s];
      float b1 = s + 1 < S ? nxt[s + 1] : NEG_INF;
      float b2 = (s + 2 < S && ext[s + 2] != blank && ext[s + 2] != ext[s]) ? nxt[s + 2] : NEG_INF;
      float v = lse3(b0, b1, b2);
      beta[t * S + s] = (v == NEG_INF) ? NEG_INF : v + logq[t * C + ext[s]];
    }
    __syncthreads();
  }
  if (tid == 0) {
    float a = alpha[(T - 1) * S + S - 1];
    float c = S >= 2 ? alpha[(T - 1) * S + S - 2] : NEG_INF;
    float lp = lse2(a, c);
    s_logp = lp;
    loss[b] = -lp;
  }
  __syncthreads();
  if (!grad) return;
  const float logp = s_logp;
  float* gz = grad + (long long)b * Tmax * C;
  for (int i = T * C + tid; i < Tmax * C; i += blockDim.x) gz[i] = 0.f;      // frames beyond this sample's length
  if (logp == NEG_INF) {                                                    // no valid alignment (T_b too short): loss = +inf
    for (int i = tid; i < T * C; i += blockDim.x) gz[i] = 0.f;
    return;
  }

  // gradient, frame by frame (block-cooperative: occupancy scatter, then a block reduction for the softmax chain)
  __shared__ float red[32];
  for (int t = 0; t < T; ++t) {
    // occupancy of class k = sum over the extended-label positions s that carry k, in position order (no atomics: the
    // blank and repeated letters occur at several positions, and a fixed order keeps the gradient bitwise repeatable)
    for (int k = tid; k < C; k += blockDim.x) {
      float o = 0.f;
      for (int s = 0; s < S; ++s) {
        if (ext[s] != k) continue;
        float ab = alpha[t * S + s] + beta[t * S + s];
        if (ab != NEG_INF) o += expf(ab - 2.f * logq[t * C + k] - logp);   // alpha*beta/q^2/P  (beta includes one q)
      }
      occ[k] = o;
    }
    __syncthreads();
    // g_u[k] = q - q*occ' where occ' = sum alpha*beta/(q^2 P) ... so occupancy/P expressed relative to q:
    //   dL/du_k = q_k - (1/P) sum_s alpha_t(s) beta_t(s) / q_k = q_k - q_k * occ[k]
    float partial = 0.f;
    for (int k = tid; k < C; k += blockDim.x) {
      float q = expf(logq[t * C + k]);
      float gu = q - q * occ[k];
      float p = q * (1.f + (float)C * CTC_EPS) - CTC_EPS;
      if (p < 0.f) p = 0.f;
      float gp = gu / (p + CTC_EPS);
      occ[k] = gp;                      // reuse as dL/dp
      partial += p * gp;
    }
    float dot = sg_block_sum(partial, red);
    for (int k = tid; k < C; k += blockDim.x) {
      float q = expf(logq[t * C + k]);
      float p = q * (1.f + (float)C * CTC_EPS) - CTC_EPS;
      if (p < 0.f) p = 0.f;
      gz[t * C + k] = p * (occ[k] - dot);
    }
    __syncthreads();
  }
}

// Allow Kernel `cap` bytes of dynamic shared memory, once per device: the attribute is a cap (a launch asks for what it uses),
// so it is not set again on every launch.  Devices >= 64 are not cached and set it every time.
template <auto Kernel>
static cudaError_t allow_dynamic_smem(const sg_ctx* ctx, int cap) {
  static std::atomic<unsigned long long> done{0};
  const unsigned long long bit = ctx->device < 64 ? 1ull << ctx->device : 0ull;
  if (bit && (done.load() & bit)) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
  if (e == cudaSuccess) done.fetch_or(bit);
  return e;
}

static int ctc_launch(sg_ctx* ctx, const float* logits, const int* labels, int b, int t, int c, int l, const int* input_len,
                      const int* label_len, float* loss, float* grad_logits, const char* who) {
  SG_REQUIRE(ctx && logits && labels && loss, "%s: NULL", who);
  SG_REQUIRE(b >= 0 && t > 0 && c > 1 && l >= 0, "%s: bad sizes", who);
  SG_REQUIRE(input_len || label_len || t >= l, "%s: %d frames cannot emit %d labels", who, t, l);
  if (b == 0) return SG_OK;
  int S = 2 * l + 1;
  size_t smem = sizeof(float) * ((size_t)t * c + 2 * (size_t)t * S + c) + sizeof(int) * S;
  SG_REQUIRE(smem <= 200 * 1024, "%s: T*C too large for shared memory (%zu bytes)", who, smem);
  if (smem > 48 * 1024) SG_CHECK_CUDA(allow_dynamic_smem<k_ctc>(ctx, 200 * 1024));
  sg_launch(ctx, k_ctc, b, 128, smem, logits, labels, t, c, l, input_len, label_len, loss, grad_logits);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

extern "C" int sg_ctc(sg_ctx* ctx, const float* logits, const int* labels, int b, int t, int c, int l, float* loss,
                      float* grad_logits) {
  return ctc_launch(ctx, logits, labels, b, t, c, l, nullptr, nullptr, loss, grad_logits, "sg_ctc");
}

/* ragged batch: per-sample frame counts input_len[b] <= t_max and label counts label_len[b] <= l_max (device int32) */
extern "C" int sg_ctc_ragged(sg_ctx* ctx, const float* logits, const int* labels, int b, int t_max, int c, int l_max,
                             const int* input_len, const int* label_len, float* loss, float* grad_logits) {
  SG_REQUIRE(input_len && label_len, "sg_ctc_ragged: NULL length arrays");
  return ctc_launch(ctx, logits, labels, b, t_max, c, l_max, input_len, label_len, loss, grad_logits, "sg_ctc_ragged");
}

// ---------------------------------------------------------------------------------------------------
// Reading words back: R's per-frame probabilities, the greedy (best-path) CTC decoding and the edit distance to a reference.
// Conventions of k_ctc: blank = C-1, per-sample frame counts T_b <= Tmax in a rectangular [b, Tmax, C] layout.
// ---------------------------------------------------------------------------------------------------
#define SOFTMAX_ROWS_PER_BLOCK 8

// y = softmax(x) over rows of C fp32 values (the reference's Dense(activation='softmax'), net_architecture.py:55); one warp
// per row (warp_softmax_row, the first stage of k_ctc)
__global__ void k_softmax_rows(const float* __restrict__ x, long long rows, int C, float* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * SOFTMAX_ROWS_PER_BLOCK + (threadIdx.x >> 5);
  if (r >= rows) return;
  warp_softmax_row(x + r * C, C, lane, [&](int k, float p) { y[r * C + k] = p; });
}

// One chunk of a block-scan compaction: the exclusive offset of this thread among the block's flagged threads (warps in
// order, then lanes) and the chunk's total.  cnt[nwarps] holds the per-warp counts; one __syncthreads after they are
// written, and the caller syncs before the next chunk rewrites them.
static __device__ __forceinline__ int block_exclusive_offset(bool flag, int* cnt, int lane, int warp, int nwarps, int* chunk) {
  const unsigned int bal = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) cnt[warp] = __popc(bal);
  __syncthreads();
  int off = __popc(bal & ((1u << lane) - 1u)), total = 0;
  for (int w = 0; w < nwarps; ++w) {
    if (w < warp) off += cnt[w];
    total += cnt[w];
  }
  *chunk = total;
  return off;
}

// Greedy decoding of one sample per CTA: best class of every frame t < T_b (ties -> lowest index), repeats merged, blanks
// dropped (a blank between two equal letters keeps both).  The emitted letters are compacted in frame order with a block
// scan.  dynamic smem: best[Tmax] (int) | logmax[Tmax] (float)
#define DECODE_THREADS 256
__global__ void __launch_bounds__(DECODE_THREADS) k_ctc_greedy_decode(const float* __restrict__ probs, int Tmax, int C,
                                                                      const int* __restrict__ input_len, int* __restrict__ decoded,
                                                                      int* __restrict__ decoded_len, float* __restrict__ neg_sum_log) {
  extern __shared__ float sm[];
  int* best = reinterpret_cast<int*>(sm);
  float* logmax = sm + Tmax;
  __shared__ int warp_cnt[DECODE_THREADS / 32];
  __shared__ float red[32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = DECODE_THREADS / 32;
  const int T = sample_frames(input_len, b, 0, Tmax);
  const float* p = probs + (long long)b * Tmax * C;
  const int blank = C - 1;

  // per-frame argmax: one warp per frame; each lane keeps its first maximum, the warp reduction prefers the lower index
  for (int t = warp; t < T; t += nwarps) {
    float v = NEG_INF;
    int idx = C;
    for (int k = lane; k < C; k += 32) {
      const float q = p[(long long)t * C + k];
      if (q > v || idx == C) { v = q; idx = k; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, v, o);
      const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
    if (lane == 0) {
      best[t] = idx;
      logmax[t] = logf(v + CTC_EPS);
    }
  }
  __syncthreads();

  // score: each thread sums its frames in frame order, then a fixed-shape block reduction -- bit-reproducible
  float part = 0.f;
  for (int t = tid; t < T; t += DECODE_THREADS) part += logmax[t];
  const float total = sg_block_sum(part, red);

  // compaction: emit[t] = best[t] != blank && best[t] != best[t-1]; exclusive block scan chunk by chunk
  int* out = decoded + (long long)b * Tmax;
  int base = 0;
  for (int t0 = 0; t0 < T; t0 += DECODE_THREADS) {
    const int t = t0 + tid;
    const int a = t < T ? best[t] : blank;
    const bool emit = t < T && a != blank && (t == 0 || best[t - 1] != a);
    int chunk;
    const int off = block_exclusive_offset(emit, warp_cnt, lane, warp, nwarps, &chunk);
    if (emit) out[base + off] = a;
    base += chunk;
    __syncthreads();                   // warp_cnt is rewritten by the next chunk
  }
  for (int t = base + tid; t < Tmax; t += DECODE_THREADS) out[t] = -1;
  if (tid == 0) {
    decoded_len[b] = base;
    neg_sum_log[b] = 0.f - total;      // 0 - x: an empty sum gives +0
  }
}

// length of a -1 padded row: the run of leading non-negative entries (sg_label_lengths), one warp
__device__ __forceinline__ int leading_nonneg(const int* row, int n, int lane) {
  for (int j0 = 0; j0 < n; j0 += 32) {
    const int j = j0 + lane;
    const unsigned int neg = __ballot_sync(0xffffffffu, j < n && row[j] < 0);
    if (neg) return j0 + __ffs(neg) - 1;
  }
  return n;
}

// Levenshtein distance, one warp per sample: Myers' bit-parallel algorithm (Hyyro's global-distance form) with the reference
// as the <= 64-symbol pattern in one 64-bit word, and the hypothesis as the text (any length).  The match mask of a
// hypothesis symbol comes from two ballots over the reference held one symbol per lane (j and j + 32).  Every lane runs the
// same (uniform) recurrence.  totals (optional) += {sum dist, sum reference length, exact matches, samples}: integer atomics,
// one per block and counter, so the result does not depend on the order.
#define EDIT_MAX_REF 64
#define EDIT_THREADS 256
__global__ void __launch_bounds__(EDIT_THREADS) k_edit_distance(const int* __restrict__ hyp, const int* __restrict__ hyp_len,
                                                                int hyp_stride, const int* __restrict__ ref,
                                                                const int* __restrict__ ref_len, int ref_stride, int nb,
                                                                int* __restrict__ dist, long long* __restrict__ totals) {
  __shared__ long long s_tot[EDIT_THREADS / 32][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * (EDIT_THREADS / 32) + warp;
  long long d = 0, m = 0, exact = 0, one = 0;
  if (b < nb) {
    const int* h = hyp + (long long)b * hyp_stride;
    const int* r = ref + (long long)b * ref_stride;
    int n = hyp_len ? hyp_len[b] : leading_nonneg(h, hyp_stride, lane);
    int mm = ref_len ? ref_len[b] : leading_nonneg(r, ref_stride, lane);
    n = n < 0 ? 0 : (n > hyp_stride ? hyp_stride : n);
    mm = mm < 0 ? 0 : (mm > ref_stride ? ref_stride : mm);
    int score = mm;
    if (mm == 0) {
      score = n;
    } else {
      const bool has_lo = lane < mm, has_hi = lane + 32 < mm;
      const int r_lo = has_lo ? r[lane] : 0, r_hi = has_hi ? r[lane + 32] : 0;
      const unsigned long long high = 1ull << (mm - 1);
      unsigned long long pv = ~0ull, mv = 0ull;
      for (int i = 0; i < n; ++i) {
        const int c = h[i];
        const unsigned long long eq = (unsigned long long)__ballot_sync(0xffffffffu, has_lo && r_lo == c) |
                                      ((unsigned long long)__ballot_sync(0xffffffffu, has_hi && r_hi == c) << 32);
        const unsigned long long xv = eq | mv;
        const unsigned long long xh = (((eq & pv) + pv) ^ pv) | eq;
        unsigned long long ph = mv | ~(xh | pv);
        unsigned long long mh = pv & xh;
        if (ph & high) ++score;
        else if (mh & high) --score;
        ph = (ph << 1) | 1ull;         // row 0 of the table grows by one per hypothesis symbol
        mh <<= 1;
        pv = mh | ~(xv | ph);
        mv = ph & xv;
      }
    }
    if (lane == 0) dist[b] = score;
    d = score; m = mm; exact = score == 0; one = 1;
  }
  if (!totals) return;
  if (lane == 0) {
    s_tot[warp][0] = d; s_tot[warp][1] = m; s_tot[warp][2] = exact; s_tot[warp][3] = one;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    long long s = 0;
    for (int w = 0; w < EDIT_THREADS / 32; ++w) s += s_tot[w][threadIdx.x];
    if (s) atomicAdd(reinterpret_cast<unsigned long long*>(totals + threadIdx.x), (unsigned long long)s);
  }
}

extern "C" int sg_softmax_rows(sg_ctx* ctx, const float* x, long long rows, int c, float* y) {
  SG_REQUIRE(ctx && x && y, "sg_softmax_rows: NULL");
  SG_REQUIRE(rows >= 0 && c >= 2, "sg_softmax_rows: bad sizes (rows %lld, c %d)", rows, c);
  if (rows == 0) return SG_OK;
  const long long blocks = (rows + SOFTMAX_ROWS_PER_BLOCK - 1) / SOFTMAX_ROWS_PER_BLOCK;
  SG_REQUIRE(blocks <= 0x7fffffffLL, "sg_softmax_rows: %lld rows", rows);
  sg_launch(ctx, k_softmax_rows, (unsigned int)blocks, 32 * SOFTMAX_ROWS_PER_BLOCK, 0, x, rows, c, y);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

extern "C" int sg_ctc_greedy_decode(sg_ctx* ctx, const float* probs, int b, int t_max, int c, const int* input_len,
                                    int* decoded, int* decoded_len, float* neg_sum_log) {
  SG_REQUIRE(ctx && probs && decoded && decoded_len && neg_sum_log, "sg_ctc_greedy_decode: NULL");
  SG_REQUIRE(b >= 0 && t_max >= 1 && c >= 2, "sg_ctc_greedy_decode: bad sizes (b %d, t_max %d, c %d)", b, t_max, c);
  const size_t smem = (size_t)t_max * (sizeof(int) + sizeof(float));
  SG_REQUIRE(smem <= 200 * 1024, "sg_ctc_greedy_decode: t_max %d too large for shared memory", t_max);
  if (b == 0) return SG_OK;
  if (smem > 48 * 1024) SG_CHECK_CUDA(allow_dynamic_smem<k_ctc_greedy_decode>(ctx, 200 * 1024));
  sg_launch(ctx, k_ctc_greedy_decode, b, DECODE_THREADS, smem, probs, t_max, c, input_len, decoded, decoded_len, neg_sum_log);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

extern "C" int sg_edit_distance(sg_ctx* ctx, const int* hyp, const int* hyp_len, int hyp_stride, const int* ref,
                                const int* ref_len, int ref_stride, int b, int* dist, long long* totals) {
  SG_REQUIRE(ctx && hyp && ref && dist, "sg_edit_distance: NULL");
  SG_REQUIRE(b >= 0 && hyp_stride >= 0 && ref_stride >= 0, "sg_edit_distance: bad sizes (b %d, hyp %d, ref %d)", b, hyp_stride,
             ref_stride);
  SG_REQUIRE(ref_stride <= EDIT_MAX_REF, "sg_edit_distance: references of up to %d symbols (got rows of %d)", EDIT_MAX_REF,
             ref_stride);
  if (b == 0) return SG_OK;
  sg_launch(ctx, k_edit_distance, sg_div_up(b, EDIT_THREADS / 32), EDIT_THREADS, 0, hyp, hyp_len, hyp_stride, ref, ref_len,
            ref_stride, b, dist, totals);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

// ---------------------------------------------------------------------------------------------------
// CTC prefix beam search (K.ctc_decode(greedy=False) / tf.nn.ctc_beam_search_decoder with the default scorer), one sample
// per CTA, the beam state in shared memory.
//   x_t = log-softmax(log(p_t + 1e-7)) over the C classes [TF-SEMANTICS: Keras feeds log(y_pred + 1e-7) to the decoder, which
//   treats its input as logits], i.e. log((p + eps) / (1 + C eps)) as in k_ctc.
//   A beam is a prefix: (log P_blank, log P_label), their total, its parent (the kept beam one symbol shorter, or -1) and its
//   last symbol.  At frame t every kept beam b of rank r offers its continuation (candidate index r C + C - 1) and its
//   extensions by c < C - 1 (index r C + c) whose prefix is not already kept -- a kept prefix b + c is a kept beam with parent
//   b and last symbol c, found in a W x C child table.  The beam_width largest totals are kept, ties to the lower index;
//   candidates of total -inf are never kept.  The selection is a radix select on orderable 64-bit (total, ~index) keys with
//   8-bit digits (integer histogram counters only), the kept candidates are ranked by counting; fp32 sums in a fixed order,
//   so the result is bit-reproducible.
//   Back-pointers (old rank << 8 | emitted symbol or 0xFF) go to the caller's scratch [b, Tmax, W]; path k is the beam of
//   rank k, read back from the last frame.  merge_repeated merges consecutive equal symbols of the written path [TF-SEMANTICS].
// dynamic smem: cand[W * C] (float) | child[W * C] (int8)
// ---------------------------------------------------------------------------------------------------
#define BEAM_THREADS 256
#define BEAM_MAX_W 128
#define BEAM_MAX_C 128
#define BEAM_NO_SYMBOL 0xFF

// the bits of s as an unsigned whose order is the float order: larger float -> larger unsigned
static __device__ __forceinline__ unsigned int ordered_bits(float s) {
  const unsigned int u = __float_as_uint(s);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ unsigned long long beam_key(float s, int pos) {             // larger total, then lower index
  return ((unsigned long long)ordered_bits(s) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned int)pos);
}

// x[k] = log-softmax(log(p[k] + eps)) over the C <= 128 classes of one frame, one warp, the row in registers
static __device__ __forceinline__ void frame_log_softmax(const float* p, int C, int lane, float* x) {
  float lp[BEAM_MAX_C / 32];
  float m = NEG_INF;
#pragma unroll
  for (int j = 0; j < BEAM_MAX_C / 32; ++j) {
    const int k = lane + 32 * j;
    lp[j] = k < C ? logf(p[k] + CTC_EPS) : NEG_INF;
    m = fmaxf(m, lp[j]);
  }
  m = sg_warp_max(m);
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < BEAM_MAX_C / 32; ++j)
    if (lane + 32 * j < C) s += expf(lp[j] - m);
  const float ls = logf(sg_warp_sum(s));
#pragma unroll
  for (int j = 0; j < BEAM_MAX_C / 32; ++j)
    if (lane + 32 * j < C) x[lane + 32 * j] = (lp[j] - m) - ls;
}

// One digit of a radix select, warp 0: scan the 256-bin histogram from the top for the bin that holds the need-th largest
// key (lane l owns bins 255 - 8l .. 248 - 8l).  One lane writes that bin's digit, the number of keys in the bins above it and
// the bin's count.  Returns the lane's inclusive count: the histogram's total on lane 31.
static __device__ __forceinline__ int radix_pick_digit(const int* hist, int need, int lane, int* digit, int* above, int* count) {
  int cnt[8], sum = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    cnt[j] = hist[255 - 8 * lane - j];
    sum += cnt[j];
  }
  int inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  const int exc = inc - sum;
  const unsigned int hit = __ballot_sync(0xffffffffu, exc < need && need <= inc);
  if (hit && lane == __ffs(hit) - 1) {
    int ab = exc, sel = -1, c = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {                     // unrolled: cnt stays in registers
      if (sel >= 0) continue;
      if (ab + cnt[j] >= need) {
        sel = j;
        c = cnt[j];
      } else {
        ab += cnt[j];
      }
    }
    *digit = 255 - 8 * lane - sel;
    *above = ab;
    *count = c;
  }
  return inc;
}

__global__ void __launch_bounds__(BEAM_THREADS) k_ctc_beam_decode(const float* __restrict__ probs, int Tmax, int C,
                                                                  const int* __restrict__ input_len, int W, int top_paths,
                                                                  int merge_repeated, int* __restrict__ decoded,
                                                                  int* __restrict__ decoded_len, float* __restrict__ log_prob,
                                                                  unsigned short* bp) {
  extern __shared__ float sm[];
  float* cand = sm;
  signed char* child = reinterpret_cast<signed char*>(sm + W * C);
  __shared__ float s_x[BEAM_MAX_C];
  __shared__ float s_pb[2][BEAM_MAX_W], s_pl[2][BEAM_MAX_W], s_tot[2][BEAM_MAX_W];
  __shared__ int s_last[2][BEAM_MAX_W], s_par[2][BEAM_MAX_W];
  __shared__ float s_npb[BEAM_MAX_W], s_npl[BEAM_MAX_W];
  __shared__ int s_contrank[BEAM_MAX_W], s_sel[BEAM_MAX_W], s_order[BEAM_MAX_W], s_len[BEAM_MAX_W];
  __shared__ unsigned long long s_selkey[BEAM_MAX_W];
  __shared__ int s_hist[256];
  __shared__ int s_nsel, s_digit, s_above, s_count, s_total;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = sample_frames(input_len, b, 0, Tmax);
  const float* p = probs + (long long)b * Tmax * C;
  unsigned short* bpb = bp + (long long)b * Tmax * W;
  const int blank = C - 1;

  for (int i = tid; i < W * C; i += BEAM_THREADS) child[i] = -1;
  if (tid == 0) {                                     // t = 0: the empty prefix, P_blank = 1, P_label = 0
    s_pb[0][0] = 0.f; s_pl[0][0] = NEG_INF; s_tot[0][0] = 0.f; s_last[0][0] = -1; s_par[0][0] = -1;
  }
  int nb = 1, cur = 0;
  __syncthreads();

  for (int t = 0; t < T; ++t) {
    const int nxt = cur ^ 1;
    if (warp == 0) frame_log_softmax(p + (long long)t * C, C, lane, s_x);   // the frame's log-probabilities
    __syncthreads();

    // candidates: cand[r C + c] = total of the extension of beam r by c, or of r's continuation at c = blank
    const int n = nb * C;
    for (int i = tid; i < n; i += BEAM_THREADS) {
      const int r = i / C, c = i - r * C;
      float v;
      if (c == blank) {
        const int last = s_last[cur][r], par = s_par[cur][r];
        const float npb = s_tot[cur][r] + s_x[blank];
        float npl = NEG_INF;
        if (last >= 0) {
          const float xl = s_x[last];
          npl = s_pl[cur][r] + xl;
          if (par >= 0) {                             // the parent's mass moves into this prefix by emitting `last`
            const float prev = last == s_last[cur][par] ? s_pb[cur][par] : s_tot[cur][par];
            npl = lse2(npl, prev + xl);
          }
        }
        s_npb[r] = npb;
        s_npl[r] = npl;
        v = lse2(npb, npl);
      } else if (child[i] >= 0) {
        v = NEG_INF;                                  // prefix already kept: its continuation accounts for it
      } else {
        v = s_x[c] + (c == s_last[cur][r] ? s_pb[cur][r] : s_tot[cur][r]);
      }
      cand[i] = v;
    }
    __syncthreads();

    // radix select of the W largest keys: digits of the total (4 passes), then of the index (bits 31..16 of ~index are all
    // ones as n <= 2^14); stops as soon as every key with the chosen prefix is kept.  kept <=> key >= prefix.
    unsigned long long prefix = 0ull, mask = 0ull;
    int need = W;
    bool keep_all = false;
    for (int pass = 0; pass < 6; ++pass) {
      const int sh = pass < 4 ? 56 - 8 * pass : 8 * (5 - pass);
      if (pass == 4) {
        prefix |= 0xFFFF0000ull;
        mask |= 0xFFFF0000ull;
      }
      for (int i = tid; i < 256; i += BEAM_THREADS) s_hist[i] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += BEAM_THREADS) {
        const float v = cand[i];
        if (v == NEG_INF) continue;
        const unsigned long long key = beam_key(v, i);
        if ((key & mask) == prefix) atomicAdd(&s_hist[(int)((key >> sh) & 0xFFull)], 1);
      }
      __syncthreads();
      if (warp == 0) {
        const int inc = radix_pick_digit(s_hist, need, lane, &s_digit, &s_above, &s_count);
        if (lane == 31) s_total = inc;
      }
      __syncthreads();
      if (pass == 0 && s_total <= need) {             // W or fewer live candidates: all kept
        keep_all = true;
        break;
      }
      need -= s_above;
      prefix |= (unsigned long long)s_digit << sh;
      mask |= 0xFFull << sh;
      if (s_count == need) break;
    }

    if (tid == 0) s_nsel = 0;
    __syncthreads();
    for (int i = tid; i < n; i += BEAM_THREADS) {     // gather (any order: the rank below does not depend on it)
      const float v = cand[i];
      if (v == NEG_INF) continue;
      const unsigned long long key = beam_key(v, i);
      if (keep_all || key >= prefix) {
        const int slot = atomicAdd(&s_nsel, 1);
        s_sel[slot] = i;
        s_selkey[slot] = key;
      }
    }
    __syncthreads();
    const int nk = s_nsel;
    for (int i = tid; i < nk; i += BEAM_THREADS) {    // rank = number of larger keys (keys are distinct)
      const unsigned long long k = s_selkey[i];
      int rank = 0;
      for (int j = 0; j < nk; ++j) rank += s_selkey[j] > k;
      s_order[rank] = s_sel[i];
    }
    for (int i = tid; i < nb; i += BEAM_THREADS) s_contrank[i] = -1;
    __syncthreads();
    for (int k = tid; k < nk; k += BEAM_THREADS) {
      const int pos = s_order[k];
      if (pos % C == blank) s_contrank[pos / C] = k;  // new rank of old beam r's continuation
    }
    for (int j = tid; j < nb; j += BEAM_THREADS)      // forget the old child table
      if (s_par[cur][j] >= 0) child[s_par[cur][j] * C + s_last[cur][j]] = -1;
    __syncthreads();
    for (int k = tid; k < nk; k += BEAM_THREADS) {    // the new beams, in rank order
      const int pos = s_order[k], r = pos / C, c = pos - r * C;
      const float v = cand[pos];
      int par, last;
      if (c == blank) {
        const int op = s_par[cur][r];
        s_pb[nxt][k] = s_npb[r];
        s_pl[nxt][k] = s_npl[r];
        last = s_last[cur][r];
        par = op >= 0 ? s_contrank[op] : -1;
      } else {
        s_pb[nxt][k] = NEG_INF;
        s_pl[nxt][k] = v;
        last = c;
        par = s_contrank[r];
      }
      s_tot[nxt][k] = v;
      s_last[nxt][k] = last;
      s_par[nxt][k] = par;
      if (par >= 0) child[par * C + last] = (signed char)k;
      bpb[(long long)t * W + k] = (unsigned short)((r << 8) | (c == blank ? BEAM_NO_SYMBOL : c));
    }
    __syncthreads();
    nb = nk;
    cur = nxt;
  }

  // path k = beam of rank k, walked back from the last frame: once to count, once to write
  for (int k = tid; k < top_paths; k += BEAM_THREADS) {
    int len = 0;
    if (k < nb) {
      int r = k, after = -1;
      for (int t = T - 1; t >= 0; --t) {
        const unsigned int e = bpb[(long long)t * W + r];
        const int sym = (int)(e & 0xFFu);
        if (sym != BEAM_NO_SYMBOL) {
          if (!merge_repeated || sym != after) ++len;
          after = sym;
        }
        r = (int)(e >> 8);
      }
      int* out = decoded + ((long long)k * gridDim.x + b) * Tmax;
      int j = len;
      r = k;
      after = -1;
      for (int t = T - 1; t >= 0; --t) {
        const unsigned int e = bpb[(long long)t * W + r];
        const int sym = (int)(e & 0xFFu);
        if (sym != BEAM_NO_SYMBOL) {
          if (!merge_repeated || sym != after) out[--j] = sym;
          after = sym;
        }
        r = (int)(e >> 8);
      }
    }
    s_len[k] = len;
    decoded_len[(long long)k * gridDim.x + b] = len;
    log_prob[(long long)b * top_paths + k] = k < nb ? s_tot[cur][k] : NEG_INF;
  }
  __syncthreads();
  for (int k = 0; k < top_paths; ++k) {
    int* out = decoded + ((long long)k * gridDim.x + b) * Tmax;
    for (int i = s_len[k] + tid; i < Tmax; i += BEAM_THREADS) out[i] = -1;
  }
}

extern "C" size_t sg_ctc_beam_decode_scratch_bytes(int b, int t_max, int beam_width) {
  if (b <= 0 || t_max <= 0 || beam_width <= 0) return 0;
  return (size_t)b * (size_t)t_max * (size_t)beam_width * sizeof(unsigned short);
}

extern "C" int sg_ctc_beam_decode(sg_ctx* ctx, const float* probs, int b, int t_max, int c, const int* input_len, int beam_width,
                                  int top_paths, int merge_repeated, int* decoded, int* decoded_len, float* log_prob,
                                  void* scratch, size_t scratch_bytes) {
  SG_REQUIRE(ctx && probs && decoded && decoded_len && log_prob, "sg_ctc_beam_decode: NULL");
  SG_REQUIRE(b >= 0 && t_max >= 1 && c >= 2 && c <= BEAM_MAX_C, "sg_ctc_beam_decode: bad sizes (b %d, t_max %d, c %d <= %d)", b,
             t_max, c, BEAM_MAX_C);
  SG_REQUIRE(beam_width >= 1 && beam_width <= BEAM_MAX_W, "sg_ctc_beam_decode: beam_width %d not in [1, %d]", beam_width,
             BEAM_MAX_W);
  SG_REQUIRE(top_paths >= 1 && top_paths <= beam_width, "sg_ctc_beam_decode: top_paths %d not in [1, beam_width %d]", top_paths,
             beam_width);
  if (b == 0) return SG_OK;
  const size_t need = sg_ctc_beam_decode_scratch_bytes(b, t_max, beam_width);
  SG_REQUIRE(scratch && scratch_bytes >= need, "sg_ctc_beam_decode: scratch of %zu bytes for %d x %d back-pointers, got %zu", need,
             b, t_max, scratch_bytes);
  const size_t smem = (size_t)beam_width * c * (sizeof(float) + 1);
  // the kernel's ~11 KB of static shared memory counts against the 48 KB default too: allow the largest dynamic size
  SG_CHECK_CUDA(allow_dynamic_smem<k_ctc_beam_decode>(ctx, (int)((size_t)BEAM_MAX_W * BEAM_MAX_C * (sizeof(float) + 1))));
  sg_launch(ctx, k_ctc_beam_decode, b, BEAM_THREADS, smem, probs, t_max, c, input_len, beam_width, top_paths, merge_repeated,
            decoded, decoded_len, log_prob, (unsigned short*)scratch);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

// ---------------------------------------------------------------------------------------------------
// Lexicon (closed-vocabulary) decoding: the CTC log-likelihood of every (sample, word) pair, and each sample's best words.
//   scores[b, v] = log p(lexicon[v] | x_b) with x_t = log-softmax(log(p_t + 1e-7)) over the C classes, as in
//   k_ctc_beam_decode: minus K.ctc_batch_cost of the pair [TF-SEMANTICS].  Forward (alpha) recursion in the log domain with
//   lse2 / lse3, no beta and no gradient.  One CTA per (sample, tile of LEX_WORDS words): the sample's frame table x[T_b, C]
//   is built in shared memory once and read by every word of the tile; one warp per word, extended-label state s on lane s
//   and lane s - 32, states s - 1 and s - 2 by warp shuffles.  A word that cannot fit in T_b frames (L + adjacent repeats >
//   T_b) or holds a symbol outside [0, C - 1) scores -inf without running the recursion; with T_b = 0 the empty word
//   scores 0.  Each score is one warp's fixed sequence of operations: bit-reproducible.
//   dynamic smem: x[Tmax * C] (float)
// ---------------------------------------------------------------------------------------------------
#define LEX_THREADS 256
#define LEX_WORDS 64
#define LEX_MAX_L 31
#define LEX_MAX_C 128
#define LEX_MAX_TOPK 128
#define LEX_MAX_SMEM (200 * 1024)
static_assert(LEX_MAX_C <= BEAM_MAX_C, "frame_log_softmax holds up to BEAM_MAX_C classes");

__global__ void __launch_bounds__(LEX_THREADS) k_ctc_lexicon_scores(const float* __restrict__ probs, int Tmax, int C,
                                                                    const int* __restrict__ input_len,
                                                                    const int* __restrict__ lexicon,
                                                                    const int* __restrict__ lex_len, int V, int Lmax,
                                                                    int tiles, float* __restrict__ scores) {
  extern __shared__ float x[];
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = LEX_THREADS / 32;
  const unsigned int full = 0xffffffffu;
  const int T = sample_frames(input_len, b, 0, Tmax);
  const float* p = probs + (long long)b * Tmax * C;
  const int blank = C - 1;

  for (int t = warp; t < T; t += nwarps)              // the frame table, one warp per frame
    frame_log_softmax(p + (long long)t * C, C, lane, x + t * C);
  __syncthreads();

  const int v_end = min(V, (tile + 1) * LEX_WORDS);
  for (int v = tile * LEX_WORDS + warp; v < v_end; v += nwarps) {
    int L = lex_len[v];
    L = L < 0 ? 0 : (L > Lmax ? Lmax : L);
    const int sym = lane < L ? lexicon[(long long)v * Lmax + lane] : blank;      // letter j on lane j (L <= 31)
    const int before = __shfl_up_sync(full, sym, 1);
    const unsigned int rep = __ballot_sync(full, lane >= 1 && lane < L && sym == before);
    const unsigned int bad = __ballot_sync(full, lane < L && (sym < 0 || sym >= blank));
    float* out = scores + (long long)b * V + v;
    if (bad || L + __popc(rep) > T) {                 // no alignment: exactly -inf
      if (lane == 0) *out = NEG_INF;
      continue;
    }
    if (T == 0) {                                     // the empty word (L = 0 here) over no frames
      if (lane == 0) *out = 0.f;
      continue;
    }
    // state s: blank for even s, letter (s - 1) / 2 for odd s; lane holds s = lane (lo) and s = lane + 32 (hi).  The skip
    // s - 2 -> s is allowed for a letter that differs from the letter before it: letter j = (s - 1) / 2 >= 1, bit j of rep clear.
    const int S = 2 * L + 1;
    const int odd = lane & 1, j_lo = lane >> 1, j_hi = 16 + (lane >> 1);
    const int l_lo = __shfl_sync(full, sym, j_lo), l_hi = __shfl_sync(full, sym, j_hi);
    const int e_lo = odd ? l_lo : blank, e_hi = odd ? l_hi : blank;
    const bool in_lo = lane < S, in_hi = lane + 32 < S;
    const bool skip_lo = odd && j_lo >= 1 && !((rep >> j_lo) & 1u), skip_hi = odd && !((rep >> j_hi) & 1u);
    float a_lo = (lane < 2 && in_lo) ? x[e_lo] : NEG_INF, a_hi = NEG_INF;
    if (S <= 32) {                                    // warp-uniform: words of up to 15 letters use the lo half only
      for (int t = 1; t < T; ++t) {
        const float u1 = __shfl_up_sync(full, a_lo, 1), u2 = __shfl_up_sync(full, a_lo, 2);
        const float v3 = lse3(a_lo, lane >= 1 ? u1 : NEG_INF, skip_lo ? u2 : NEG_INF);
        a_lo = (in_lo && v3 != NEG_INF) ? v3 + x[t * C + e_lo] : NEG_INF;
      }
    } else {
      for (int t = 1; t < T; ++t) {
        const float u1 = __shfl_up_sync(full, a_lo, 1), u2 = __shfl_up_sync(full, a_lo, 2);
        const float h1 = __shfl_up_sync(full, a_hi, 1), h2 = __shfl_up_sync(full, a_hi, 2);
        const float w1 = __shfl_sync(full, a_lo, 31), w2 = __shfl_sync(full, a_lo, 30 + (lane & 1));   // states 31 and 30/31
        const float n_lo = lse3(a_lo, lane >= 1 ? u1 : NEG_INF, skip_lo ? u2 : NEG_INF);
        const float n_hi = lse3(a_hi, lane >= 1 ? h1 : w1, skip_hi ? (lane >= 2 ? h2 : w2) : NEG_INF);
        const float* xt = x + t * C;
        a_lo = (in_lo && n_lo != NEG_INF) ? n_lo + xt[e_lo] : NEG_INF;
        a_hi = (in_hi && n_hi != NEG_INF) ? n_hi + xt[e_hi] : NEG_INF;
      }
    }
    // log p = lse2(alpha[S - 1], alpha[S - 2]) at the last frame, in k_ctc's order
    const int s1 = S - 1, s2 = S - 2 < 0 ? 0 : S - 2;
    const float f1 = __shfl_sync(full, s1 < 32 ? a_lo : a_hi, s1 & 31);
    const float f2 = __shfl_sync(full, s2 < 32 ? a_lo : a_hi, s2 & 31);
    if (lane == 0) *out = lse2(f1, S >= 2 ? f2 : NEG_INF);
  }
}

// Top-k words of every sample, one CTA per row of V scores: radix select of the k largest orderable 32-bit keys (four 8-bit
// digits, integer histogram counters in shared memory, warp-aggregated), then the keys above the threshold and the first
// tied keys in index order are compacted with a block scan, and the <= 128 survivors are ranked by counting.  Equal scores go
// to the lower word index; -inf is ranked like any other score (-0 and +0 are equal).  The chosen words are gathered from
// the lexicon in the same launch.
__device__ __forceinline__ unsigned int lex_key(float s) { return ordered_bits(s == 0.f ? 0.f : s); }

__global__ void __launch_bounds__(LEX_THREADS) k_ctc_lexicon_topk(const float* __restrict__ scores, int V,
                                                                  const int* __restrict__ lexicon,
                                                                  const int* __restrict__ lex_len, int Lmax, int K,
                                                                  int* __restrict__ decoded, int* __restrict__ decoded_len,
                                                                  float* __restrict__ log_prob, int* __restrict__ index) {
  __shared__ int s_hist[256];
  __shared__ int s_digit, s_above, s_count;
  __shared__ int s_wcnt[2][LEX_THREADS / 32];
  __shared__ unsigned int s_key[LEX_MAX_TOPK];
  __shared__ int s_idx[LEX_MAX_TOPK], s_order[LEX_MAX_TOPK];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = LEX_THREADS / 32;
  const unsigned int full = 0xffffffffu;
  const float* row = scores + (long long)b * V;

  // the K-th largest key: after pass p its top 8(p + 1) bits are `prefix`; need = how many keys with that prefix are kept
  unsigned int prefix = 0u, mask = 0u;
  int need = K;
  for (int pass = 0; pass < 4; ++pass) {
    const int sh = 24 - 8 * pass;
    for (int i = tid; i < 256; i += LEX_THREADS) s_hist[i] = 0;
    __syncthreads();
    for (int i0 = 0; i0 < V; i0 += LEX_THREADS) {
      const int i = i0 + tid;
      const unsigned int key = i < V ? lex_key(row[i]) : 0u;
      const int bin = (i < V && (key & mask) == prefix) ? (int)((key >> sh) & 0xFFu) : 256;
      const unsigned int peers = __match_any_sync(full, bin);
      if (bin < 256 && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], __popc(peers));
    }
    __syncthreads();
    if (warp == 0) radix_pick_digit(s_hist, need, lane, &s_digit, &s_above, &s_count);
    __syncthreads();
    need -= s_above;
    prefix |= (unsigned int)s_digit << sh;
    mask |= 0xFFu << sh;
    if (s_count == need) break;                       // every key with this prefix is kept
  }

  // compaction in index order: keys whose prefix is above, and the first `need` keys with the prefix
  int base_eq = 0, base_sel = 0;
  for (int i0 = 0; i0 < V && base_sel < K; i0 += LEX_THREADS) {
    const int i = i0 + tid;
    const unsigned int key = i < V ? lex_key(row[i]) : 0u;
    const bool gt = i < V && (key & mask) > prefix, eq = i < V && (key & mask) == prefix;
    int eq_chunk, chunk;
    const int eq_before = base_eq + block_exclusive_offset(eq, s_wcnt[0], lane, warp, nwarps, &eq_chunk);
    const bool take = gt || (eq && eq_before < need);
    const int off = base_sel + block_exclusive_offset(take, s_wcnt[1], lane, warp, nwarps, &chunk);
    if (take) {
      s_key[off] = key;
      s_idx[off] = i;
    }
    base_eq += eq_chunk;
    base_sel += chunk;
    __syncthreads();                                  // s_wcnt is rewritten by the next chunk
  }
  for (int k = tid; k < K; k += LEX_THREADS) {        // rank = larger keys + equal keys of lower index (kept in index order)
    const unsigned int key = s_key[k];
    int rank = 0;
    for (int j = 0; j < K; ++j) rank += s_key[j] > key || (s_key[j] == key && j < k);
    s_order[rank] = k;
  }
  __syncthreads();
  for (int k = warp; k < K; k += nwarps) {            // path k: one warp gathers the word
    const int v = s_idx[s_order[k]];
    int L = lex_len[v];
    L = L < 0 ? 0 : (L > Lmax ? Lmax : L);
    const long long o = (long long)k * gridDim.x + b;
    int* out = decoded + o * Lmax;
    for (int i = lane; i < Lmax; i += 32) out[i] = i < L ? lexicon[(long long)v * Lmax + i] : -1;
    if (lane == 0) {
      decoded_len[o] = L;
      log_prob[(long long)b * K + k] = row[v];
      index[(long long)b * K + k] = v;
    }
  }
}

extern "C" int sg_ctc_lexicon_scores(sg_ctx* ctx, const float* probs, int b, int t_max, int c, const int* input_len,
                                     const int* lexicon, const int* lex_len, int v, int l_max, float* scores) {
  SG_REQUIRE(ctx, "sg_ctc_lexicon_scores: NULL context");
  SG_REQUIRE(b >= 0 && t_max >= 1 && v >= 0, "sg_ctc_lexicon_scores: bad sizes (b %d, t_max %d, v %d)", b, t_max, v);
  SG_REQUIRE(c >= 2 && c <= LEX_MAX_C, "sg_ctc_lexicon_scores: c %d not in [2, %d]", c, LEX_MAX_C);
  SG_REQUIRE(l_max >= 0 && l_max <= LEX_MAX_L, "sg_ctc_lexicon_scores: words of up to %d symbols (got rows of %d)", LEX_MAX_L,
             l_max);
  const size_t smem = (size_t)t_max * c * sizeof(float);
  SG_REQUIRE(smem <= LEX_MAX_SMEM, "sg_ctc_lexicon_scores: t_max %d x c %d frame table (%zu bytes) exceeds %d bytes of shared "
             "memory", t_max, c, smem, LEX_MAX_SMEM);
  if (b == 0 || v == 0) return SG_OK;                            // nothing to read or write
  SG_REQUIRE(probs && lex_len && scores && (lexicon || l_max == 0), "sg_ctc_lexicon_scores: NULL");
  const long long tiles = (v + LEX_WORDS - 1) / LEX_WORDS;
  SG_REQUIRE((long long)b * tiles <= 0x7fffffffLL, "sg_ctc_lexicon_scores: %d samples x %lld word tiles", b, tiles);
  SG_CHECK_CUDA(allow_dynamic_smem<k_ctc_lexicon_scores>(ctx, LEX_MAX_SMEM));    // the largest frame table
  sg_launch(ctx, k_ctc_lexicon_scores, (unsigned int)(b * tiles), LEX_THREADS, smem, probs, t_max, c, input_len, lexicon, lex_len,
            v, l_max, (int)tiles, scores);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}

extern "C" int sg_ctc_lexicon_topk(sg_ctx* ctx, const float* scores, int b, int v, const int* lexicon, const int* lex_len,
                                   int l_max, int top_paths, int* decoded, int* decoded_len, float* log_prob, int* index) {
  SG_REQUIRE(ctx, "sg_ctc_lexicon_topk: NULL context");
  SG_REQUIRE(b >= 0 && v >= 0 && l_max >= 0, "sg_ctc_lexicon_topk: bad sizes (b %d, v %d, l_max %d)", b, v, l_max);
  SG_REQUIRE(top_paths >= 1 && top_paths <= v && top_paths <= LEX_MAX_TOPK,
             "sg_ctc_lexicon_topk: top_paths %d not in [1, min(v %d, %d)]", top_paths, v, LEX_MAX_TOPK);
  if (b == 0) return SG_OK;
  SG_REQUIRE(scores && lex_len && decoded_len && log_prob && index && (l_max == 0 || (lexicon && decoded)),
             "sg_ctc_lexicon_topk: NULL");
  sg_launch(ctx, k_ctc_lexicon_topk, b, LEX_THREADS, 0, scores, v, lexicon, lex_len, l_max, top_paths, decoded, decoded_len,
            log_prob, index);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}
