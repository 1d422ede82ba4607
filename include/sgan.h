/* libsgan -- C ABI of the B200-native ScrabbleGAN train-step kernels.
 *
 * The reference (UtkuKaradeniz/scrabble-gan) has NO native/FFI layer: its hot path is Python calling
 * TensorFlow ops.  Every entry point below therefore replaces the TF op(s) a given reference line
 * dispatches to; the citation after each prototype is `file:line` under /root/reference/src/bigacgan
 * (SURVEY.md section 2.2 maps K1..K21 to these).  The host side stays Python and binds these with ctypes
 * (scrabble-gan_b200/_abi.py); see INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  Every pointer is a DEVICE pointer unless stated.
 *   - every function returns int: SG_OK (0) or a negative error class; text via sg_last_error().
 *   - all launches are asynchronous on the context's stream; nothing synchronises except sg_ctx_sync.
 *   - no hidden allocation: scratch memory is passed in by the caller.
 *   - layouts are TensorFlow's: activations NHWC contiguous, Conv2D kernels HWIO, Conv2DTranspose
 *     kernels (kh,kw,Cout,Cin), Dense kernels (in,out), labels int32.
 *   - "operand" tensors (inputs of convolutions) are SG_F32 or SG_BF16; reductions, residual streams,
 *     gradients of parameters and optimizer state are always fp32.
 */
#ifndef SGAN_H_
#define SGAN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sg_ctx sg_ctx;

enum { SG_OK = 0, SG_ERR_ARG = -1, SG_ERR_CUDA = -2, SG_ERR_UNSUPPORTED = -3 };
enum { SG_F32 = 0, SG_BF16 = 1 };
#define SG_MAX_TAPS 16

/* ---- context ------------------------------------------------------------------------------------ */
int sg_version(void);
const char* sg_last_error(void);
int sg_ctx_create(int device, void* cuda_stream, sg_ctx** out);
int sg_ctx_destroy(sg_ctx* ctx);
int sg_ctx_set_stream(sg_ctx* ctx, void* cuda_stream);
int sg_ctx_sync(sg_ctx* ctx);
/* zero `bytes` of device memory on the context's stream (cudaMemsetAsync: no kernel launch) */
int sg_zero(sg_ctx* ctx, void* ptr, size_t bytes);
long long sg_ctx_launch_count(sg_ctx* ctx);      /* kernels launched through this context so far */
/* speed mode (bf16 runs): the fp32 1x1 projections of the non-local block take their products on bf16 warp-level tensor
 * ops (fp32 accumulate) instead of exact FFMA; off by default */
int sg_ctx_set_speed_mode(sg_ctx* ctx, int on);
/* tensor-core convolutions: when the last wave of output tiles of a launch would leave most SMs idle, the k-range of each of its
 * tiles is split over several CTAs, which exchange fp32 partial accumulators through the context's workspace and add them in a
 * fixed order (results stay bit-reproducible run to run).  On by default. */
int sg_ctx_set_conv_split_tail(sg_ctx* ctx, int on);
int sg_sizeof_conv_desc(void);                    /* sizeof(sg_conv_desc): layout guard for FFI mirrors */

/* ---- convolution family (K1-K8) ------------------------------------------------------------------
 * One descriptor covers Conv2D forward, its dgrad (a conv with swapped channel roles), Conv2DTranspose
 * (phase-decomposed: one call per output phase, strided output placement) and its dgrad (strided input
 * sampling).  out[n, oy*out_sy+out_py, ox*out_sx+out_px, co] (+)= act( bias[co] +
 *      sum_t sum_ci in[n, oy*in_sy+tap_dy[t], ox*in_sx+tap_dx[t], ci] * W_t[ci,co] ) * (mask > 0)
 * with W_t[ci,co] = w_master[tap_w_off[t] + ci*w_ci_stride + co*w_co_stride]; out-of-range input = 0.
 * Replaces tf Conv2D / Conv2DBackpropInput / Conv2DTranspose: resnet_ops.py:57,65,69,98,103,109;
 * net_architecture.py:28-49,283; arch_ops.py:38-65. */
typedef struct sg_conv_desc {
  int n;
  int in_h, in_w, c_in;
  int out_h, out_w, c_out;
  int grid_h, grid_w;
  int in_sy, in_sx;
  int out_sy, out_sx, out_py, out_px;
  int ntaps;
  int tap_dy[SG_MAX_TAPS];
  int tap_dx[SG_MAX_TAPS];
  long long tap_w_off[SG_MAX_TAPS];
  long long w_ci_stride, w_co_stride;
  int in_dt, out_dt;
  int relu;
  int accumulate;
  int mask_dt;
} sg_conv_desc;

/* exact-fp32 direct convolution (any shape; used for Cin=1 / Cout=1 edge layers and as the fp32 mode) */
int sg_conv_fwd_simt(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const float* w_master,
                     const float* bias, const void* mask, void* out);
/* filter gradient of the conv described by d: dw_master[tap_w_off[t] + ci*.. + co*..] += sum in * dy.
 * `dy` is indexed like `out` (dtype d->out_dt).  Replaces Conv2DBackpropFilter (tapes, data_utils.py:450-467). */
int sg_conv_wgrad_simt(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master);

/* tcgen05/TMEM/TMA implicit-GEMM path (operands bf16 or fp32-as-tf32, fp32 accumulate in TMEM) */
int sg_conv_tc_supported(const sg_conv_desc* d);
size_t sg_conv_packed_weight_elems(const sg_conv_desc* d);     /* c_out * ntaps * c_in */
int sg_conv_pack_weights(sg_ctx* ctx, const sg_conv_desc* d, const float* w_master, void* w_packed);
/* several packing jobs (<= 32: e.g. all forward filters of a network after an optimizer step) in ONE launch; descs / w_master /
 * w_packed are HOST arrays of length njobs; sg_conv_pack_multi_supported says whether a filter qualifies. */
int sg_conv_pack_multi_supported(const sg_conv_desc* d, const float* w_master);
int sg_conv_pack_weights_multi(sg_ctx* ctx, int njobs, const sg_conv_desc* const* descs, const float* const* w_master,
                               void* const* w_packed);
int sg_conv_fwd_tc(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed,
                   const float* bias, const void* mask, void* out);
/* out = epilogue( conv(d, in, w_packed) + conv1x1(d2, in2, w_packed2) ): the shortcut of a ResNet block
 * (resnet_ops.py:109-114) accumulated in TMEM as extra k-blocks of the main conv -- no second pass over the output.
 * d2: 1x1, stride 1, same batch / pixel grid / c_out / operand dtype; both filters packed (sg_conv_pack_weights). */
/* Host-only planning query (no GPU needed): the N tile (columns per output tile), the number of output tiles and the k-split of
 * the tiles of a partial last wave that sg_conv_fwd_tc would use for this descriptor on a device with num_sms SMs. */
int sg_conv_tc_plan(const sg_conv_desc* d, int num_sms, int split_tail_enabled, int* bn_out, int* split_out, int* tiles_out);
/* sg_conv_fwd_tc plus a rank-1 term in the epilogue: out[p, c] = conv(in)[p, c] + bias[c] + r1_x[p] * r1_w[c] (before ReLU /
 * mask).  This is the 1x1 shortcut conv of a residual block whose input has ONE channel (D.B1 on the raw image,
 * resnet_ops.py:107-110): an outer product, folded into the main conv instead of a launch that re-reads and re-writes the
 * whole output.  r1_x: fp32 [n, out_h, out_w]; r1_w: fp32 [c_out]; unit output stride only. */
int sg_conv_fwd_tc_rank1(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed, const float* bias,
                         const void* mask, void* out, const float* r1_x, const float* r1_w);
/* The output phases of a Conv2DTranspose forward (resnet_ops.py:57,69; phase-decomposed: no zero-stuffed MACs) as ONE launch.
 * descs[i] (1..4) are the per-phase descriptors: same tensors, pixel grid and dtypes, different taps and output offsets
 * (out_py, out_px); the filter is read in place from the bf16 mirror of the master weights.  A stride-2 3x3 transposed conv
 * is 4 + 2 + 2 + 1 taps = one launch of 4x the tiles instead of four launches that each fill a fraction of the SMs. */
int sg_conv_fwd_tc_phases(sg_ctx* ctx, int nphase, const sg_conv_desc* const* descs, const void* in, const void* w_mirror_bf16,
                          const float* bias, void* out);
int sg_conv_fwd_tc_dual(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_packed,
                        const sg_conv_desc* d2, const void* in2, const void* w_packed2, const float* bias,
                        const void* mask, void* out);
/* the same launch reading the filter IN PLACE from a bf16 mirror of the master weights (identical indexing): no packing
 * pass.  HWIO forward convs use the mirror as an N-major B operand, dgrads / transposed-conv phases as a K-major one. */
int sg_conv_tc_direct_supported(const sg_conv_desc* d);
int sg_conv_fwd_tc_direct(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* w_mirror_bf16,
                          const float* bias, const void* mask, void* out);
size_t sg_conv_wgrad_tc_workspace(const sg_conv_desc* d, int num_sms);
int sg_conv_wgrad_tc(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master,
                     void* workspace, size_t workspace_bytes);
/* the same launch also producing the layer's BIAS gradient (BiasAddGrad of resnet_ops.py:65,98,103 / net_architecture.py:28-49):
 * db[c_out] (and db2 when not NULL: the bias of the block's shortcut conv, which sees the same upstream gradient) += column
 * sums of dy, computed on the tensor cores as dy^T . 1 by extra units that reuse the dy tiles.  Plain Conv2D filter
 * gradients only (the pixel grid must cover dy exactly once). */
int sg_conv_wgrad_tc_bias(sg_ctx* ctx, const sg_conv_desc* d, const void* in, const void* dy, float* dw_master,
                          float* db, float* db2);
/* 1 when those extra units fit into the idle CTA slots of the launch's last wave (the bias gradient is then free), 0 when
 * they would open another wave (a separate column sum is faster: use sg_colsum). */
int sg_conv_wgrad_tc_bias_fits(sg_ctx* ctx, const sg_conv_desc* d);

/* ---- element-wise glue --------------------------------------------------------------------------- */
/* relu_out = relu(x), copy_out = x, both cast to out_dt (either may be NULL).  resnet_ops.py:97,101 */
int sg_act_prep(sg_ctx* ctx, const float* x, long long n, void* relu_out, void* copy_out, int out_dt);
/* out (+)= dy * (act > 0)   (ReLU backward) */
int sg_mask_mul(sg_ctx* ctx, const float* dy, const void* act, int act_dt, void* out, int out_dt,
                long long n, int accumulate);
/* out = a*x + b*y (y may be NULL)   -- residual adds, resnet_ops.py:73,114 */
int sg_axpby(sg_ctx* ctx, float a, const float* x, float b, const float* y, float* out, long long n);
/* out = (*sigma)*a + x  (x may be NULL => out = sigma*a)   -- arch_ops.py:67 */
int sg_scale_add(sg_ctx* ctx, const float* sigma, const float* a, const float* x, float* out, long long n);
int sg_tanh_fwd(sg_ctx* ctx, const float* x, float* y, long long n);                  /* net_architecture.py:289 */
int sg_tanh_bwd(sg_ctx* ctx, const float* dy, const float* y, float* dx, long long n);
/* x[r, :] *= w[r] */
int sg_scale_rows(sg_ctx* ctx, float* x, const float* w, int rows, long long cols);
/* out[0] (+)= sum a*b */
/* x[i, :] *= up[i] * mult for the samples i < n of a batch-first tensor [n, per_sample] (fp32 / bf16; per_sample % 8 == 0).
 * Samples with factor 1 are skipped, samples with factor 0 are zero-filled without being read.  Used by the merged
 * discriminator backward: the fake half of the batch is back-propagated ONCE with a constant upstream weight; the filter
 * gradients of the D loss then need the per-sample weights of that loss (hinge: 0 or 1). */
int sg_scale_samples(sg_ctx* ctx, void* x, int dt, int n, long long per_sample, const float* up, float mult);
int sg_dot(sg_ctx* ctx, const float* a, const float* b, long long n, float* out, int accumulate);
/* out[c] (+)= sum_r x[r,c]   (bias gradients) */
int sg_colsum(sg_ctx* ctx, const void* x, int dt, long long rows, int cols, float* out, int accumulate);
int sg_cast(sg_ctx* ctx, const float* x, void* out, int out_dt, long long n);

/* ---- pooling (K11) ------------------------------------------------------------------------------- */
int sg_avgpool2_fwd(sg_ctx* ctx, const float* x, int n, int h, int w, int c, float* out);   /* resnet_ops.py:106,113 */
int sg_avgpool2_bwd(sg_ctx* ctx, const float* dout, int n, int h, int w, int c, void* dx, int dx_dt);
int sg_maxpool_fwd(sg_ctx* ctx, const void* x, int dt, int n, int h, int w, int c, int ph, int pw,
                   void* out);                                                          /* net_architecture.py:29-47; arch_ops.py:47,58 */
int sg_maxpool_bwd(sg_ctx* ctx, const float* dout, const void* x, int x_dt, int n, int h, int w, int c,
                   int ph, int pw, int relu_mask, void* dx, int dx_dt);
int sg_gap_relu_fwd(sg_ctx* ctx, const float* x, int n, long long hw, int c, float* out);   /* net_architecture.py:249-250,340-341 */
int sg_gap_relu_bwd(sg_ctx* ctx, const float* dfeat, const float* x, int n, long long hw, int c, float* dx);

/* ---- batch norm / conditional batch norm (K9, K10) ------------------------------------------------
 * resnet_ops.py:13-28 (CBN), net_architecture.py:42,46,281 (BN).  Statistics are exchanged as raw sums
 * so that the caller can all-reduce them across data-parallel replicas between the two calls. */
size_t sg_bn_stats_scratch_bytes(long long rows, int c);
int sg_bn_stats(sg_ctx* ctx, const float* x, long long rows, int c, float* sums /*[2c]*/, void* scratch,
                size_t scratch_bytes);
int sg_bn_finalize(sg_ctx* ctx, const float* sums, double count, int c, float eps, float momentum,
                   float* mean, float* rstd, float* moving_mean, float* moving_var);
int sg_bn_infer_prepare(sg_ctx* ctx, const float* moving_mean, const float* moving_var, int c, float eps,
                        float* mean, float* rstd);
/* out = act( (x-mean)*rstd*gamma + beta ); gamma/beta are [n,c] (gb_stride=c) or [c] (gb_stride=0), NULL => 1 / 0 */
int sg_bn_apply(sg_ctx* ctx, const float* x, int n, long long hw, int c, const float* mean,
                const float* rstd, const float* gamma, const float* beta, long long gb_stride, int relu,
                void* out, int out_dt);
/* s1[n,c] = sum_hw dyr, s2[n,c] = sum_hw dyr*xhat, dyr = dy*(act>0) (act NULL => no mask) */
int sg_bn_bwd_reduce(sg_ctx* ctx, const float* dy, const void* act, int act_dt, const float* x, int n,
                     long long hw, int c, const float* mean, const float* rstd, float* s1, float* s2);
/* ab[0:c] = sum_n gamma*s1, ab[c:2c] = sum_n gamma*s2  (per-channel terms of the BN backward; all-reduce me) */
int sg_bn_bwd_combine(sg_ctx* ctx, const float* s1, const float* s2, const float* gamma,
                      long long gb_stride, int n, int c, float* ab);
/* dx (+)= rstd*(gamma*dyr - [ab0 + xhat*ab1]/count) [* (x > 0) if mask_by_x]
 * (batch terms dropped when use_batch_terms==0: inference-mode BN, SURVEY Q5) */
int sg_bn_bwd_apply(sg_ctx* ctx, const float* dy, const void* act, int act_dt, const float* x, int n,
                    long long hw, int c, const float* mean, const float* rstd, const float* gamma,
                    long long gb_stride, const float* ab, double count, int use_batch_terms, int mask_by_x,
                    void* dx, int dx_dt, int accumulate);

/* ---- small cross-replica exchanges over NVLink peer memory (data-parallel sync-BN / loss sums) -------------------
 * peer_bufs[r] = base address of rank r's exchange buffer (sg_peer_buffer_bytes() bytes of SYMMETRIC memory, zeroed
 * once before the first call) as mapped in THIS process.  All ranks must issue the same sequence of exchange calls; the
 * call sequence number lives in the buffer itself (device resident), so the launches can be replayed from a CUDA graph.
 * One launch: publish -> flag peers -> wait -> sum in rank order (bit-identical on all ranks).
 * Replaces a NCCL all-reduce of <= sg_peer_max_payload_bytes() bytes. */
size_t sg_peer_buffer_bytes(void);
size_t sg_peer_max_payload_bytes(void);
int sg_peer_allreduce_sum(sg_ctx* ctx, void* data, int n, int is_f64, const unsigned long long* peer_bufs, int world,
                          int rank);
/* Gradient buckets (data parallel, SURVEY 8e exchange point 3): SUM all-reduce of a large fp32 vector that every replica keeps in
 * peer-mapped (symmetric) memory, moved by the COPY ENGINES over NVLink -- the SMs stay with the step's compute kernels, which
 * an SM-based collective running beside 148-CTA persistent kernels cannot offer (measured: overlapping NCCL's all-reduce with
 * the backward pass gained nothing).  Reduce-scatter + all-gather, pull side: barrier; memcpy MY shard of every peer's bucket
 * into staging; add in rank order (k_bucket_reduce: bit-identical on every replica); barrier; memcpy every peer's reduced shard;
 * barrier.  All on ctx's stream: enqueue it on a stream of its own and it overlaps with whatever the compute stream runs.
 *   g_ptrs[r]   = replica r's bucket as mapped in this process (g_ptrs[rank] == g)
 *   flag_bufs   = a sg_peer_buffer_bytes() exchange buffer per replica, used by no other stream (barrier flags)
 *   staging     = (world - 1) * sg_peer_bucket_shard(n, world) floats of local scratch
 *   use_sms     = 1: the same exchange with kernels reading the peers over NVLink (k_bucket_pull_reduce / k_bucket_gather,
 *                 4 CTAs per SM) -- for a bucket whose all-reduce is exposed, i.e. nothing is left to overlap with */
long long sg_peer_bucket_shard(long long n, int world);
int sg_peer_barrier(sg_ctx* ctx, const unsigned long long* peer_bufs, int world, int rank);
int sg_peer_bucket_allreduce(sg_ctx* ctx, float* g, long long n, float* staging, const unsigned long long* g_ptrs,
                             const unsigned long long* flag_bufs, int world, int rank, int use_sms);
/* sync-BN forward statistics in one launch after the per-block partial sums: stage-2 reduction + exchange + mean /
 * rstd / moving-average finalisation (FusedBatchNormV3 training statistics, resnet_ops.py:14-17) */
int sg_bn_stats_partial(sg_ctx* ctx, const float* x, long long rows, int c, void* scratch, size_t scratch_bytes,
                        int* nblocks_out);
int sg_bn_finalize_peer(sg_ctx* ctx, const float* partial, int nblocks, int c, double count_total, float eps,
                        float momentum, float* sums_out, float* mean, float* rstd, float* moving_mean,
                        float* moving_var, const unsigned long long* peer_bufs, int world, int rank);

/* ---- small dense GEMM (K14): C (+)= op(A) op(B) + bias;  row-major, fp32 -------------------------- */
int sg_gemm(sg_ctx* ctx, int trans_a, int trans_b, int m, int n, int k, const float* a, int lda,
            const float* b, int ldb, float* c, int ldc, const float* bias, int accumulate);

/* ---- filter bank (K13) -- arch_ops.py:84-90; net_architecture.py:230-231,260-271 ------------------
 * out[b, k%4, 4l + k/2048, (k%2048)/4] = sum_j z[b*z_stride + j] * bank[y[b,l], j, k]   (bit-exact index map) */
int sg_filterbank_fwd(sg_ctx* ctx, const float* z, int z_stride, const int* y, int b, int l, int vocab,
                      const float* bank, float* out);
int sg_filterbank_bwd(sg_ctx* ctx, const float* dout, const float* z, int z_stride, const int* y, int b,
                      int l, int vocab, const float* bank, float* dbank /*overwritten*/,
                      float* dz0 /*dz0[b*dz_stride + j], j<32; or NULL*/, int dz_stride);

/* ---- non-local block core (K12) -- arch_ops.py:51-61: o = softmax(theta phi^T) g, no scaling ------- */
int sg_attn_fwd(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv,
                int dk, int dv, float* o, float* lse);
int sg_attn_bwd(sg_ctx* ctx, const float* theta, const float* phi, const float* g, const float* o,
                const float* lse, const float* d_o, int n, int q, int kv, int dk, int dv, float* dtheta,
                float* dphi, float* dg);

/* tensor-core variant for the speed (bf16) mode: theta.phi^T in tf32, P.g in bf16 (mma.sync register chaining), fp32
 * softmax; same arguments and results within bf16 tolerance.  scratch: n*q floats (D = rowsum(dO o O)). */
int sg_attn_tc_supported(int q, int kv, int dk, int dv);
int sg_attn_fwd_tc(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv,
                   int dk, int dv, float* o, float* lse);
int sg_attn_bwd_tc(sg_ctx* ctx, const float* theta, const float* phi, const float* g, const float* o,
                   const float* lse, const float* d_o, int n, int q, int kv, int dk, int dv, float* dtheta,
                   float* dphi, float* dg, float* scratch);

/* 1x1 projections of the non-local block, one pass over the pixels per data-flow step (arch_ops.py:38-46,55-57,63-67).
 * C = 64 channels, dk = 8, dv = 32; x, dx, og, out, dout are [rows,64]; theta/phi_f [rows,8]; g_f, o, d_o [rows,32];
 * kernels w_theta, w_phi [64,8], w_g [64,32], w_o [32,64] (1x1 HWIO).  Filter gradients are accumulated (+=). */
int sg_nonlocal_proj_fwd(sg_ctx* ctx, const float* x, long long rows, const float* w_theta, const float* w_phi,
                         const float* w_g, float* theta, float* phi_f, float* g_f);
/* og = o . w_o (kept for d sigma = <dout, og>);  out = (*sigma) * og + x */
int sg_nonlocal_out_fwd(sg_ctx* ctx, const float* o, long long rows, const float* w_o, const float* sigma,
                        const float* x, float* og, float* out);
/* d_o = (*sigma) * dout . w_o^T;  dw_o += (*sigma) * o^T . dout  (dw_o may be NULL) */
int sg_nonlocal_out_bwd(sg_ctx* ctx, const float* dout, const float* o, long long rows, const float* w_o,
                        const float* sigma, float* d_o, float* dw_o);
/* dx += dtheta . w_theta^T + dphi_f . w_phi^T + dg_f . w_g^T;  dw_* += x^T . d*  (all three dw_* or none) */
int sg_nonlocal_proj_bwd(sg_ctx* ctx, const float* x, const float* dtheta, const float* dphi_f, const float* dg_f,
                         long long rows, const float* w_theta, const float* w_phi, const float* w_g, float* dx,
                         float* dw_theta, float* dw_phi, float* dw_g);

/* ---- CTC (K15) -- net_architecture.py:55-72: softmax -> log(p+1e-7) -> tf.nn.ctc_loss --------------
 * loss[b] = -log p(labels_b | x_b); grad_logits = d loss / d (Dense pre-activations), blank = c-1 */
int sg_ctc(sg_ctx* ctx, const float* logits, const int* labels, int b, int t, int c, int l, float* loss,
           float* grad_logits);
/* ragged batch -- K.ctc_batch_cost's own interface (net_architecture.py:57-72 passes per-sample input_length / label_length):
 * input_len[b] <= t_max frames and label_len[b] <= l_max labels per sample (device int32); logits / labels / grad keep the
 * rectangular [b, t_max, c] / [b, l_max] layout; frames beyond a sample's length get a zero gradient; a sample without any
 * valid alignment gets loss = +inf and a zero gradient. */
int sg_ctc_ragged(sg_ctx* ctx, const float* logits, const int* labels, int b, int t_max, int c, int l_max,
                  const int* input_len, const int* label_len, float* loss, float* grad_logits);

/* ---- reading words back with the recogniser (same conventions as sg_ctc: blank = c-1, [b, t_max, c] layout) -------------
 * sg_softmax_rows: y = softmax(x) over rows of c fp32 values -- the reference's Dense(activation='softmax') output
 * (net_architecture.py:55), i.e. what a Keras user feeds to K.ctc_decode. */
int sg_softmax_rows(sg_ctx* ctx, const float* x, long long rows, int c, float* y);
/* Replaces K.ctc_decode(greedy=True) / tf.nn.ctc_greedy_decoder(merge_repeated=True): per frame t < input_len[b] (NULL: all
 * t_max frames; clamped to [0, t_max]) the most probable class (ties: lowest index), repeats merged, blanks dropped.
 * decoded [b, t_max] int32 padded with -1, decoded_len [b], neg_sum_log[b] = -sum_t log(max_c probs[b,t,c] + 1e-7) (Keras'
 * log_prob; [TF-SEMANTICS]).  Deterministic.  t_max <= 25600. */
int sg_ctc_greedy_decode(sg_ctx* ctx, const float* probs, int b, int t_max, int c, const int* input_len,
                         int* decoded, int* decoded_len, float* neg_sum_log);
/* Replaces K.ctc_decode(greedy=False) / tf.nn.ctc_beam_search_decoder(merge_repeated) with the default scorer: CTC prefix beam
 * search over frames t < input_len[b] (NULL: all t_max; clamped to [0, t_max]) of x = log-softmax(log(probs + 1e-7))
 * [TF-SEMANTICS], beam_width in [1, 128] kept prefixes (ties: lower candidate index), 2 <= c <= 128, 1 <= top_paths <=
 * beam_width.  Path k is the beam of rank k: decoded [top_paths, b, t_max] int32 padded with -1 (merge_repeated: consecutive
 * equal symbols merged [TF-SEMANTICS]), decoded_len [top_paths, b], log_prob [b, top_paths] = the beam's log probability
 * (-inf and length 0 beyond the live beams; 0 for the empty word of a sample without frames).  Deterministic.  scratch holds
 * the back-pointers: at least sg_ctc_beam_decode_scratch_bytes(b, t_max, beam_width) bytes. */
size_t sg_ctc_beam_decode_scratch_bytes(int b, int t_max, int beam_width);
int sg_ctc_beam_decode(sg_ctx* ctx, const float* probs, int b, int t_max, int c, const int* input_len, int beam_width,
                       int top_paths, int merge_repeated, int* decoded, int* decoded_len, float* log_prob, void* scratch,
                       size_t scratch_bytes);
/* Replaces K.ctc_batch_cost over every (sample, word) pair of a lexicon: scores [b, v] = log p(lexicon[v] | x_b), minus the
 * CTC loss of the pair, with x = log-softmax(log(probs + 1e-7)) over frames t < input_len[b] (NULL: all t_max; clamped to
 * [0, t_max]) [TF-SEMANTICS].  lexicon [v, l_max] int32 padded with -1, lex_len [v] word lengths (clamped to [0, l_max]).
 * A word that cannot fit in its sample's frames (length + adjacent repeats > frames) or holds a symbol outside [0, c - 1)
 * scores -inf; over 0 frames the empty word scores 0.  Limits: l_max <= 31, 2 <= c <= 128, t_max * c * 4 <= 200 KB.
 * Deterministic. */
int sg_ctc_lexicon_scores(sg_ctx* ctx, const float* probs, int b, int t_max, int c, const int* input_len, const int* lexicon,
                          const int* lex_len, int v, int l_max, float* scores);
/* Replaces the arg-max / top-k over the lexicon of those scores: per sample (row of scores [b, v]) the top_paths largest
 * scores, exact, equal scores to the lower word index, -inf ranked like any other score; 1 <= top_paths <= min(v, 128).
 * Path k: decoded [top_paths, b, l_max] int32 (the word, padded with -1), decoded_len [top_paths, b], log_prob [b, top_paths]
 * (its score), index [b, top_paths] (its row in the lexicon).  Deterministic. */
int sg_ctc_lexicon_topk(sg_ctx* ctx, const float* scores, int b, int v, const int* lexicon, const int* lex_len, int l_max,
                        int top_paths, int* decoded, int* decoded_len, float* log_prob, int* index);
/* Replaces tf.edit_distance(normalize=False): exact Levenshtein distance dist[b] between hyp [b, hyp_stride] and
 * ref [b, ref_stride] (int32, ref_stride <= 64).  A NULL length array means the run of leading non-negative entries
 * (sg_label_lengths).  totals (NULL or long long[4], device) is ADDED to: {sum dist, sum ref length, exact matches, samples}. */
int sg_edit_distance(sg_ctx* ctx, const int* hyp, const int* hyp_len, int hyp_stride, const int* ref, const int* ref_len,
                     int ref_stride, int b, int* dist, long long* totals);

/* ---- word augmentation for training R on its own -- replaces nothing in the reference: the HTR augmentation of the paper's
 * HTR experiments (random affine warp + thin / thick strokes).  src, dst [n, h, w] fp32 (NHWC, C = 1), out of place; h = 32.
 * widths [n] (NULL: all w) = each word's columns; dst columns >= widths[b] are copied from src bit for bit.  u [n, 7] in
 * [-1, 1) (sg_random, normal = 0) sets word b's parameters: rotation u0 * rot_deg degrees, horizontal shear u1 * shear,
 * scales 1 + u2 * scale and 1 + u3 * scale, translation (u4, u5) * translate_px; a 3x3 grey minimum if u6 < -1 + 2 p_morph,
 * a 3x3 grey maximum if u6 > 1 - 2 p_morph.  The inverse map about the word's centre (widths[b] / 2, h / 2) is sampled
 * bilinearly, coordinates clamped to the word (border replicate); the min / max leaves neighbours outside the word out.
 * Ranges >= 0, scale < 1, p_morph <= 0.5; all ranges zero copy src bit for bit.  widths live in device memory, where the
 * entry point cannot read them without a synchronisation: a width outside [1, w] makes that word's output NaN.  Draws no
 * random numbers; deterministic. */
int sg_word_augment(sg_ctx* ctx, const float* src, float* dst, int n, int h, int w, const int* widths, const float* u,
                    float rot_deg, float shear, float scale, float translate_px, float p_morph);

/* ---- GAN losses + gradient balancing (K16, K17) -- net_loss.py:4-54; data_utils.py:418-442,476-490 --
 * sums is double[SG_LOSS_NSUMS]; all-reduce it across replicas between the two calls. */
#define SG_LOSS_NSUMS 16
#define SG_LOSS_NSTATS 16
enum { SG_LOSS_HINGE = 0, SG_LOSS_NOT_SATURATING = 1 };
int sg_loss_sums(sg_ctx* ctx, int kind, int use_w, const float* d_real, const float* d_fake,
                 const float* s_real, const float* s_fake, const float* s_slot5, const float* r_fake,
                 const float* r_real, int b, double* sums);
/* up_*: per-sample upstream weights d(sum target)/d(logit) for each backward pass; stats: the 16-tuple
 * returned by train_step (data_utils.py:470-473 order). */
int sg_loss_finish(sg_ctx* ctx, int kind, int use_w, int balance, float alpha, const float* d_real,
                   const float* d_fake, const float* s_real, const float* s_fake, const float* s_slot5,
                   const float* r_fake, int b, const double* sums, float* up_d_real, float* up_d_fake_d,
                   float* up_s_real, float* up_s_fake_w, float* up_s_slot5, float* up_d_fake_g,
                   float* up_s_fake_g, float* up_r_fake_g, float* stats);

/* stand-alone forms of the reference's public loss functions: terms is float[7][b] in net_loss.py's return order
 * (d_loss, d_loss_real, d_loss_fake, g_loss, s_loss, s_loss_1, s_loss_2); s_c may be NULL for hinge. */
int sg_loss_terms(sg_ctx* ctx, int kind, const float* d_real, const float* d_fake, const float* s_a,
                  const float* s_b, const float* s_c, int b, float* terms);
/* apply_gradient_balancing (data_utils.py:476-490): g_balanced, r_balanced [b]; stds = {std(r_fake), std(g_loss)} */
int sg_grad_balance(sg_ctx* ctx, const float* r_fake, const float* g_loss, int b, float alpha,
                    float* g_balanced, float* r_balanced, float* stds);

/* Paper-faithful gradient balancing (arXiv 2003.10557 section 3.4; BASELINE north_star "std(grad_D)/std(grad_R)"): both
 * gradients are w.r.t. the generated image; out = grad_d + alpha * (std(grad_d) / std(grad_r)) * grad_r with population
 * std over all n elements.  sums is double[8] ({sum d, sum d^2, sum r, sum r^2, n, 0, 0, 0}): all-reduce it across
 * replicas between the two calls.  `stats` (may be NULL) is the step's 16-tuple, patched with the balanced losses, alpha and
 * the two stds.  The reference fork balances LOSS values instead (data_utils.py:476-490): that is sg_loss_finish. */
int sg_image_grad_balance_sums(sg_ctx* ctx, const float* grad_d, const float* grad_r, long long n, double* sums);
int sg_image_grad_balance_apply(sg_ctx* ctx, const float* grad_d, const float* grad_r, long long n, float alpha,
                                const double* sums, float* out, float* stats);

/* ---- optimizers (K19) -- main.py:25-35: Keras Adam / RMSprop --------------------------------------- */
int sg_adam(sg_ctx* ctx, float* w, const float* g, float* m, float* v, long long n, float lr_t,
            float beta1, float beta2, float eps);
/* Adam that also refreshes the bf16 mirror of the weights in the same pass */
int sg_adam_mirror(sg_ctx* ctx, float* w, const float* g, float* m, float* v, void* w_mirror_bf16, long long n,
                   float lr_t, float beta1, float beta2, float eps);
/* device-resident step size (CUDA-graph replay of the update): sg_adam_prepare sets (t >= 0) or advances (t < 0) the
 * device step counter and writes lr_t = lr sqrt(1-b2^t)/(1-b1^t); sg_adam_dev reads lr_t from lr_dev (mirror may be NULL) */
int sg_adam_prepare(sg_ctx* ctx, int* step_dev, float* lr_dev, int t, float lr, float beta1, float beta2);
int sg_adam_dev(sg_ctx* ctx, float* w, const float* g, float* m, float* v, void* w_mirror_bf16, long long n,
                const float* lr_dev, float beta1, float beta2, float eps);
/* the train step's optimizer launch (one per network): sg_adam_dev that (i) with beta1 == 0 -- the reference's setting
 * (scrabble_gan.gin:8), where Keras' m_t equals g_t -- neither reads nor writes the first-moment slot (it is then not
 * maintained), and (ii) with clear_grad overwrites the consumed gradient with zeros, so the next step needs no memset. */
int sg_adam_fused(sg_ctx* ctx, float* w, float* g, float* m, float* v, void* w_mirror_bf16, long long n, const float* lr_dev,
                  float beta1, float beta2, float eps, int clear_grad);
int sg_rmsprop(sg_ctx* ctx, float* w, const float* g, float* ms, long long n, float lr, float rho, float eps);

/* ---- spectral norm (K18) -- arch_ops.py:99-126; one power iteration from an explicit u ------------- */
int sg_spectral_norm(sg_ctx* ctx, const float* w, int rows, int cols, const float* u, int power_iteration,
                     float* w_out, float* u_out, float* sigma_out, float* scratch /* rows+cols+4 floats */);

/* ---- ragged-width batches (SURVEY 8f rank 3: words of different lengths in ONE launch, per-word SAME-padding semantics) --------
 * sg_label_lengths: lens[b] = leading labels >= 0 of a (b, l) label matrix padded with -1;  sg_mask_width: zero an NHWC tensor
 * right of every word's own width cols_per_char * lens[n] (applied to the inputs of every convolution of the generator, so that
 * a short word sees the zero padding it would see on its own);  sg_attn_fwd[_tc]_masked: the non-local block with the keys
 * beyond a word's width removed from the softmax (key j lies in column j % kv_w; kv_cols[n] columns are valid). */
int sg_label_lengths(sg_ctx* ctx, const int* labels, int b, int l, int* lens);
int sg_mask_width(sg_ctx* ctx, void* x, int dt, int n, int h, int w, int c, const int* lens, int cols_per_char);
int sg_attn_fwd_masked(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv, int dk, int dv,
                       int kv_w, const int* kv_cols, float* o, float* lse);
int sg_attn_fwd_tc_masked(sg_ctx* ctx, const float* theta, const float* phi, const float* g, int n, int q, int kv, int dk, int dv,
                          int kv_w, const int* kv_cols, float* o, float* lse);

/* ---- grouped conditional-batch-norm Dense layers (resnet_ops.py:18-26: gamma / beta = Dense(32 -> C, no bias)(z_block)) -----
 * ONE launch for all segments i < nseg (<= 16): out[n, sum c] = concat_i( z[:, z_off[i] : z_off[i] + 32] @ W_i ), W_i the (32, c[i])
 * kernel at w_base + w_off[i]; and one launch for all their filter gradients dW_i += z_slice^T @ upstream[i] ((n, c[i]) each).
 * c / z_off / w_off / upstream are HOST arrays of length nseg. */
int sg_cbn_dense_fwd(sg_ctx* ctx, const float* z, int z_stride, int n, int nseg, const int* c, const int* z_off,
                     const long long* w_off, const float* w_base, float* out);
int sg_cbn_dense_wgrad(sg_ctx* ctx, const float* z, int z_stride, int n, int nseg, const int* c, const int* z_off,
                       const long long* w_off, const float* const* upstream, float* dw_base);

/* ---- counter-based random numbers (K21; replaces tf.random.normal of data_utils.py:385) -- Philox4x32-10.  out[n] ~ U[-1,1)
 * (normal = 0) or N(0,1) (normal = 1, Box-Muller) at stream position offset + *offset_dev (offset_dev may be NULL); a given
 * offset_dev is advanced by ceil(n / 4) afterwards, so CUDA-graph replays continue the stream. */
int sg_random(sg_ctx* ctx, float* out, long long n, unsigned long long seed, unsigned long long offset,
              unsigned long long* offset_dev, int normal);

/* ---- host utility: CRC32C (Castagnoli) of a HOST buffer, chained through `crc` (start with 0).  TensorFlow checkpoints --
 * what the reference's save_weights writes (data_utils.py:346-348) -- protect tensors and index blocks with it. */
unsigned int sg_crc32c(const void* host_data, size_t n, unsigned int crc);

/* backward of the weight re-parameterisation W_sn = W / sigma (u, v constants), in place on g = dL/dW_sn:
 * g <- (g - <g, W_sn> v u^T) / sigma.  fwd_scratch is the scratch sg_spectral_norm filled for this weight (it holds the
 * un-normalised v and its inverse norm), u_hat its u_out, dot_scratch one float.  Paper-faithful option `apply_sn`:
 * in the reference spectral_norm is a kernel_regularizer nobody reads (arch_ops.py:99-126, SURVEY Q2). */
int sg_spectral_norm_bwd(sg_ctx* ctx, float* g, const float* w_sn, int rows, int cols, const float* u_hat,
                         const float* sigma, const float* fwd_scratch, float* dot_scratch);

#ifdef __cplusplus
}
#endif
#endif /* SGAN_H_ */
