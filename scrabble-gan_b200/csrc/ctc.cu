// Fused softmax -> log(p + 1e-7) -> CTC loss -> gradient w.r.t. the Dense pre-activations (K15).
// Reference: net_architecture.py:55 (Dense softmax) and :57-72 (K.ctc_batch_cost):
//     y_pred = log(softmax(z) + 1e-7);  loss = tf.nn.ctc_loss(inputs=y_pred, ...)   (which re-softmaxes its inputs)
// => effective per-frame distribution q = (p + eps) / (1 + C eps), blank = C-1, repeats merged.
// One CTA per sample; thread s owns extended-label state s (S = 2L+1); log-space alpha/beta in shared memory.
// dL/du (u = log(p+eps)) = q - occupancy/P  [tf.nn.ctc_loss gradient], chained through log and softmax to z.
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

// dynamic smem: logq[T*C] | alpha[T*S] | beta[T*S] | occ[C] | ext[S] (int)
// Ragged batches (K.ctc_batch_cost's own interface: per-sample input_length / label_length, net_architecture.py:57-72):
// input_len / label_len, when given, hold every sample's frame count T_b <= Tmax and label count L_b <= Lmax; logits / labels
// / grad keep the rectangular [b, Tmax, C] / [b, Lmax] layout, frames t >= T_b get a zero gradient.
__global__ void k_ctc(const float* __restrict__ logits, const int* __restrict__ labels, int Tmax, int C, int Lmax,
                      const int* __restrict__ input_len, const int* __restrict__ label_len, float* __restrict__ loss,
                      float* __restrict__ grad) {
  extern __shared__ float sm[];
  const int b = blockIdx.x;
  int T = input_len ? input_len[b] : Tmax, L = label_len ? label_len[b] : Lmax;
  T = T < 1 ? 1 : (T > Tmax ? Tmax : T);
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
  for (int t = warp; t < T; t += nwarps) {
    float mx = NEG_INF;
    for (int k = lane; k < C; k += 32) mx = fmaxf(mx, z[t * C + k]);
    mx = sg_warp_max(mx);
    float sum = 0.f;
    for (int k = lane; k < C; k += 32) sum += expf(z[t * C + k] - mx);
    sum = sg_warp_sum(sum);
    float inv = 1.f / sum;
    for (int k = lane; k < C; k += 32) {
      float p = expf(z[t * C + k] - mx) * inv;
      logq[t * C + k] = logf(p + CTC_EPS) - log_norm;
    }
  }
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

static int ctc_launch(sg_ctx* ctx, const float* logits, const int* labels, int b, int t, int c, int l, const int* input_len,
                      const int* label_len, float* loss, float* grad_logits, const char* who) {
  SG_REQUIRE(ctx && logits && labels && loss, "%s: NULL", who);
  SG_REQUIRE(b >= 0 && t > 0 && c > 1 && l >= 0, "%s: bad sizes", who);
  SG_REQUIRE(input_len || label_len || t >= l, "%s: %d frames cannot emit %d labels", who, t, l);
  if (b == 0) return SG_OK;
  int S = 2 * l + 1;
  size_t smem = sizeof(float) * ((size_t)t * c + 2 * (size_t)t * S + c) + sizeof(int) * S;
  SG_REQUIRE(smem <= 200 * 1024, "%s: T*C too large for shared memory (%zu bytes)", who, smem);
  if (smem > 48 * 1024) SG_CHECK_CUDA(cudaFuncSetAttribute(k_ctc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
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
// per row, max-subtracted exp and an fp32 sum -- the first stage of k_ctc
__global__ void k_softmax_rows(const float* __restrict__ x, long long rows, int C, float* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * SOFTMAX_ROWS_PER_BLOCK + (threadIdx.x >> 5);
  if (r >= rows) return;
  const float* z = x + r * C;
  float mx = NEG_INF;
  for (int k = lane; k < C; k += 32) mx = fmaxf(mx, z[k]);
  mx = sg_warp_max(mx);
  float sum = 0.f;
  for (int k = lane; k < C; k += 32) sum += expf(z[k] - mx);
  sum = sg_warp_sum(sum);
  const float inv = 1.f / sum;
  for (int k = lane; k < C; k += 32) y[r * C + k] = expf(z[k] - mx) * inv;
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
  int T = input_len ? input_len[b] : Tmax;
  T = T < 0 ? 0 : (T > Tmax ? Tmax : T);
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
    const unsigned int bal = __ballot_sync(0xffffffffu, emit);
    if (lane == 0) warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int off = base, chunk = 0;
    for (int w = 0; w < nwarps; ++w) {
      if (w < warp) off += warp_cnt[w];
      chunk += warp_cnt[w];
    }
    if (emit) out[off + __popc(bal & ((1u << lane) - 1u))] = a;
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
  if (smem > 48 * 1024)
    SG_CHECK_CUDA(cudaFuncSetAttribute(k_ctc_greedy_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
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
