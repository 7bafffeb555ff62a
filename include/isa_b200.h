/* isa_b200.h -- C ABI of libisa_sm100.so: the B200 (sm_100a) kernels of the per-pixel
 * instance-embedding hot path of Snoworday/instance-segmentation-attention.
 *
 * Conventions (they mirror the reference's one native op, the vendored SRU
 * autograd.Function that launches precompiled kernels on raw data_ptr()s:
 * /root/reference/code/lib/archs/modules/sru/cuda_functional.py:441-547):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless its
 *     name starts with h_ ; all tensors are dense and contiguous in the stated order;
 *   - the caller owns every buffer, outputs and workspace included (size queries:
 *     isa_*_workspace_bytes); the library keeps no state between calls;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*) and returns
 *     without synchronising unless stated;
 *   - return value: 0 = ok, <0 = rejected argument (ISA_ERR_*), >0 = a cudaError_t;
 *     isa_last_error() gives the message for the calling thread;
 *   - there is no CPU fallback: without a compute-capability-10.x device every
 *     compute entry point fails.
 */
#ifndef ISA_B200_H_
#define ISA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISA_ERR_BAD_ARG (-1)
#define ISA_ERR_UNSUPPORTED (-2)
#define ISA_ERR_WORKSPACE (-3)

typedef void* isa_stream_t; /* cudaStream_t */

const char* isa_last_error(void);
int isa_version(void);
int isa_num_sms(int* out);
/* Diagnostics: FP32 multiply-adds per clock per SM sustained by scalar FFMA (packed = 0) or fma.rn.f32x2 / FFMA2
 * (packed = 1) with warps_per_sm resident warps of 16 independent chains each; synchronises the device. */
int isa_selftest_fma_rate(int packed, int warps_per_sm, float sm_clock_mhz, void* scratch, float* h_fma_per_clk_per_sm);
/* Diagnostics: TMEM read rate (bytes per clock per SM) of `warps` in {4,8,16} warps issuing tcgen05.ld.32x32b.x{cols}, cols in {16,32}. */
int isa_selftest_tmem_ld_rate(int warps, int cols, float sm_clock_mhz, void* scratch, float* h_bytes_per_clk_per_sm);
/* Diagnostics: mean device time (us) of one grid-wide barrier between ctas_per_sm * num_sms co-resident CTAs
 * (variant 0: fence per thread + sleeping poll, 1: cooperative-groups style) -- the fixed cost per iteration of the
 * persistent cooperative kernels.  Synchronises the device; scratch = 8 bytes of device memory; result on the host. */
int isa_selftest_grid_barrier(int ctas_per_sm, int threads, int iters, int variant, void* scratch, float* h_us_per_barrier);

/* ------------------------------------------------------------------ discriminative loss
 * Replaces DiscriminativeLoss.forward + autograd backward:
 *   /root/reference/code/lib/losses/discriminative.py:162-188 (composite), :191-213 (class),
 *   :7-62 means, :65-95 variance, :98-132 distance, :135-147 regulariser, :149-160 q-regulariser.
 * emb        [bs][C][H][W] f32 (the NCHW tensor the network emits; no permute needed)
 * target     kind 0: u8 label map [bs][H][W], 255 = background (1 B/pixel)
 *            kind 1/2/3: dense masks [bs][K][H][W] as f32 / i64 / u8 (one-hot or soft),
 *            i.e. exactly what the reference's collate hands over (lib/dataset.py:354-376)
 * n_objects  [bs] i32 (device)
 * w_*        weights of the four terms; the shipped composite is (1, 0, 0, 0.005)
 * q_den      NULL, or a device float overriding the q-regulariser denominator int(sum(target)) of
 *            discriminative.py:153-159 (data parallel: global foreground count / world size, so that
 *            the rank-averaged loss equals the single-process loss of the whole batch)
 * out_loss [1], out_terms [4] = unweighted (var, dist, reg, qreg), out_means [bs][K][C]
 * A dense target is distilled once into a u8 label map kept in the workspace (1 byte per pixel for both passes);
 * if some pixel is not one-hot (soft / overlapping masks) the kernels keep reading the dense masks.
 * workspace  isa_disc_loss_workspace_bytes(bs,C,K,H,W) bytes; hand the SAME buffer, untouched,
 *            to isa_disc_loss_bwd (it carries the per-instance sums saved for backward).
 * Limits: 1 <= bs <= 65535, 1 <= C <= 64, 1 <= K <= 254, H*W < 2^30, norm 1 or 2 (else ISA_ERR_BAD_ARG).
 * The column-walk forward keeps 4 * (K*(CP+1) + K*(2C+1) + 256*((C+1)|1)) bytes in shared memory (CP = C rounded up to
 * 8, 16, 24, 32 or 64).  It runs for every dense target, and for a label map whose bs is above the label-map kernel's
 * co-resident CTAs.  Where that does not fit an SM those calls return ISA_ERR_UNSUPPORTED; on a B200 (232,448 B of
 * shared memory per CTA) that is C >= 54 with K above a bound that falls from 252 at C = 54 to 213 at C = 64.  Every call is checked before anything is enqueued: a refused call leaves every buffer as it was.
 */
#define ISA_TGT_LABEL_U8 0
#define ISA_TGT_DENSE_F32 1
#define ISA_TGT_DENSE_I64 2
#define ISA_TGT_DENSE_U8 3

size_t isa_disc_loss_workspace_bytes(int bs, int C, int K, int H, int W);

/* What isa_disc_loss_fwd / isa_disc_loss_bwd launch for these sizes on the current device; enqueues nothing.
 * h_plan [ISA_DISC_PLAN_LEN] host ints:
 *   0 route (ISA_DISC_ROUTE_*), 1 CP (padded channel count of the kernels' templates),
 *   2 priv of the label-map kernel (1: per-warp accumulators, bit-reproducible; 0: one CTA accumulator with shared
 *     atomics; -1: the route has no label-map kernel), 3 its CTAs per image, 4 its grid, 5 its dynamic shared memory (bytes),
 *   6 CTAs per image of the column walk (0 when the route has none), 7 its grid, 8 its dynamic shared memory,
 *   9 dynamic shared memory of the backward's prep kernel, 10 the backward's CTAs per image, 11 its dynamic shared memory.
 * Returns ISA_ERR_BAD_ARG as the forward does, and ISA_ERR_UNSUPPORTED when no route fits. */
#define ISA_DISC_ROUTE_LAB 0           /* label map: the label-map kernel alone */
#define ISA_DISC_ROUTE_COL_THEN_LAB 1  /* dense target: the column walk (which returns at once if the masks are one-hot), then the label-map kernel */
#define ISA_DISC_ROUTE_COL 2           /* the column walk alone (on a dense one-hot target: on the label map distilled from it) */
#define ISA_DISC_PLAN_LEN 12
int isa_disc_loss_plan(int target_kind, int bs, int C, int K, int H, int W, int* h_plan);

int isa_disc_loss_fwd(const float* emb, const void* target, int target_kind, const int* n_objects,
                      int bs, int C, int H, int W, int K,
                      float delta_v, float delta_d, int norm, int normalize_means,
                      float w_var, float w_dist, float w_reg, float w_q,
                      const float* q_den, float* out_loss, float* out_terms, float* out_means,
                      void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* grad_loss [1] f32 (device), grad_means [bs][K][C] or NULL, grad_emb [bs][C][H][W] out. */
int isa_disc_loss_bwd(const float* emb, const void* target, int target_kind, const int* n_objects,
                      int bs, int C, int H, int W, int K,
                      float delta_v, float delta_d, int norm, int normalize_means,
                      float w_var, float w_dist, float w_reg, float w_q,
                      const float* q_den, const float* means, const float* grad_loss, const float* grad_means,
                      float* grad_emb, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* Dense one-hot masks (kind 1..3) -> u8 label map; *not_onehot_flag (device int) is set to 1
 * when some pixel has several non-zeros or a weight other than 1; *fg_count (device u64, may be NULL) receives the
 * number of foreground pixels = int(sum(target)) of discriminative.py:153-159 for a one-hot target, so the data-parallel
 * q-regulariser denominator needs no second pass over the masks.
 * Replaces the int64 one-hot expansion of lib/dataset.py:354-376 on the device side. */
int isa_onehot_to_labels(const void* target, int target_kind, int bs, int K, int H, int W,
                         unsigned char* labels, int* not_onehot_flag, unsigned long long* fg_count, isa_stream_t stream);
/* Foreground pixels (label < K) of a u8 label map [total] -> *fg_count (device u64). */
int isa_label_fg_count(const unsigned char* labels, long long total, int K, unsigned long long* fg_count, isa_stream_t stream);

/* ------------------------------------------------------------------ embedding clustering
 * Replaces sklearn.cluster.KMeans(n_clusters=k, n_init=35, max_iter=500).fit_predict(X) as called by
 *   /root/reference/code/lib/prediction.py:72-74
 * (scikit-learn is third party, not under /root/reference; algorithm restated from scikit-learn 1.9.0:
 * sklearn/cluster/_kmeans.py:180-283 k-means++, :625-760 Lloyd loop, :1463-1563 fit,
 * _k_means_lloyd.pyx:26-211, _k_means_common.pyx:13-262; arithmetic contract: oracle/kmeans_oracle.c).
 * X           [C][ld] f32, FEATURE-major; the first n columns are the points (not modified)
 * n_ptr       device int: number of points (so the fg count never visits the host)
 * uniforms    device f64 [n_init][1 + (k-1)*n_local_trials]: the numpy RandomState(seed).random_sample
 *             stream KMeans consumes (choice for the first centre, uniform for the D^2 draws); or NULL with
 * init_centers device f32 [n_init][k][C] (array init; the data mean is subtracted like KMeans.fit does)
 * labels_out  [ld] i32 (first n valid), centers_out [k][C], inertia_out [n_init] f64, n_iter_out [n_init],
 * seed_idx_out [n_init][k] (k-means++ picks, may be NULL),
 * info        [16] i32: status (0 ok, 1 n<k, 2 non-finite input), best restart, n, Lloyd (grid) iterations run;
 *             [4..9] a coarse phase profile of the persistent Lloyd kernel as seen by CTA 0, in microseconds:
 *             E-steps, barrier after them, centre updates, barrier after them, whole loop, tail (re-run, inertia, selection);
 *             [10..15] the same for the seeding kernel: candidate search, candidate potentials, closest update, grid
 *             barriers (microseconds), then the number of scan segments and 8192-element rounds of CTA 0's searches.
 * k-means++ follows scikit-learn's float32 code path decision for decision (float64-upcast candidate distances,
 * candidates by searchsorted on the SEQUENTIAL float32 cumulative sum, float32 potentials).  E-step: packed FP32
 * (fma.rn.f32x2) or, from 33 centres on (C <= 32, k <= 128), tcgen05 MMAs as a filter with an exact pass for the pairs
 * inside the error bound -- both bit-exact with the oracle.
 */
size_t isa_kmeans_workspace_bytes(int ld, int C, int k, int n_init);

int isa_kmeans_fit(const float* X, const int* n_ptr, int ld, int C, int k, int n_init, int max_iter, double tol_rel,
                   int n_local_trials, const double* uniforms, const float* init_centers,
                   int* labels_out, float* centers_out, double* inertia_out, int* n_iter_out, int* seed_idx_out,
                   int* info, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* Foreground compaction: cls = argmax over classes (first max), fg = cls != 0, points in np.where order.
 *   /root/reference/code/lib/prediction.py:57-69
 * sem [ncls][HW] f32, emb [C][HW] f32 -> cls_map [HW] u8, Xt [C][ld] f32, fg_index [HW] i32, n_out [1]. */
size_t isa_fg_compact_workspace_bytes(int HW);

int isa_fg_compact(const float* sem, const float* emb, int ncls, int C, int HW, int ld,
                   unsigned char* cls_map, float* Xt, int* fg_index, int* n_out,
                   void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* mask[fg_index[i]] = labels[i] + 1 (uint8, 0 = background), then cv2.resize(INTER_NEAREST) of the
 * instance mask and the class map to (out_h, out_w).
 *   /root/reference/code/lib/prediction.py:76-83 (scatter), :47-50 and :105-108 (up-sampling)
 * ins_up / cls_up may be NULL. */
int isa_scatter_labels_upsample(const int* labels, const int* fg_index, const int* n_ptr,
                                const unsigned char* cls_map, int h, int w, int out_h, int out_w,
                                unsigned char* ins_small, unsigned char* ins_up, unsigned char* cls_up,
                                isa_stream_t stream);

/* ------------------------------------------------------------------ dense attention
 * Replaces ScaledDotProductAttention.forward (+ autograd backward):
 *   /root/reference/code/lib/archs/modules/utils.py:305-329
 *     attn = softmax(masked_fill(q k^T / temperature, -inf), dim=2); out = attn v
 * as called by MultiHeadAttention.forward (utils.py:193-225) with q,k,v already split per head:
 *   q [BH][Lq][d], k [BH][Lk][d], v [BH][Lk][dv] f32, BH = n_head*batch (head-major), d, dv <= 16.
 * Masks are u8, 1 = masked: key_mask [n_mask_rows][Lk] (broadcast over queries) and/or
 * full_mask [n_mask_rows][Lq][Lk]; row used for head-batch bh is bh % n_mask_rows, which equals the
 * reference's mask.repeat(n_head,1,1) without the copy.  A fully masked row yields NaN like the reference.
 * out [BH][Lq][dv]; lse2 [BH][Lq] = log2-sum-exp2 of the scaled scores (needed by bwd / probs; may be NULL).
 * Forward is a tcgen05 (TMEM accumulator) kernel fed by TMA bulk copies; operands are split into
 * bf16 hi+lo so products are fp32-accurate.  The L_q x L_k probabilities are produced only by
 * isa_attention_probs.
 * dropout_p in [0, 1) is the reference's attention-probability dropout (nn.Dropout(attn_dropout) on the softmax output,
 * utils.py:311,326), fused: the keep decision of element (bh, query, key) is a hash of (dropout_seed, bh, query, key), kept
 * probabilities are scaled by 1 / (1 - p) (p quantised to 1/65536); nothing is stored, isa_attention_bwd and
 * isa_attention_probs regenerate the same mask from the same (dropout_p, dropout_seed).  0 = no dropout (eval mode). */
size_t isa_attention_workspace_bytes(int BH, int Lq, int Lk);

int isa_attention_fwd(const float* q, const float* k, const float* v, int BH, int Lq, int Lk, int d, int dv, float temperature,
                      const unsigned char* key_mask, const unsigned char* full_mask, int n_mask_rows,
                      float dropout_p, unsigned long long dropout_seed,
                      float* out, float* lse2, void* workspace, size_t workspace_bytes, isa_stream_t stream);

int isa_attention_probs(const float* q, const float* k, const float* lse2, int BH, int Lq, int Lk, int d, float temperature,
                        const unsigned char* key_mask, const unsigned char* full_mask, int n_mask_rows,
                        float dropout_p, unsigned long long dropout_seed, float* attn, isa_stream_t stream);

int isa_attention_bwd(const float* q, const float* k, const float* v, const float* out, const float* dout, const float* lse2,
                      int BH, int Lq, int Lk, int d, int dv, float temperature,
                      const unsigned char* key_mask, const unsigned char* full_mask, int n_mask_rows,
                      float dropout_p, unsigned long long dropout_seed,
                      float* dq, float* dk, float* dv_out, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ ReNet bidirectional-GRU sweeps
 * Replaces the recurrent part of ReNet's rnn_hor / rnn_ver (nn.GRU, bidirectional):
 *   /root/reference/code/lib/archs/modules/README.md:225-256 (contract; renet.py is absent from the tree,
 *   the arithmetic is PyTorch's nn.GRU: r,z = sigmoid(..), n = tanh(W_in x + b_in + r*(W_hn h + b_hn)),
 *   h' = (1-z)*n + z*h, weight_hh_l0 (3n, n) in gate order r,z,n).
 * All tensors are token-major ("channels last"):
 *   gx    [tokens][2][3n]  x W_ih^T (+ b_ih) of both directions (one GEMM by the caller)
 *   w_hh  [2][3n][n], b_hh [2][3n]; b_ih [2][3n] or NULL when gx already carries the input-side bias
 *   out   [tokens][2n]     h_t of direction 0 in [0,n), of direction 1 (reverse sweep) in [n,2n)
 *   stash [tokens][2][4n]  r, z, n, (W_hn h + b_hn) kept for backward, or NULL for inference
 * Sequence q (0 <= q < n_seq) at step t lives at token
 *   (q / inner) * outer_tok_stride + (q % inner) * inner_tok_stride + t * t_tok_stride,
 * so a row sweep over [B][H][W] is (n_seq=B*H, T=W, inner=B*H, 0, W, 1) and a column sweep is
 * (n_seq=B*W, T=H, inner=W, H*W, 1, W).  h_0 = 0.  n_units: multiple of 4, <= 128.
 * Backward writes dgx [tokens][2][3n] (gradient of the input projection; its r,z thirds are also the
 * hidden-side gate gradients) and dghn [tokens][2][n] (hidden-side n-gate gradient r*dn_pre);
 * weight/bias gradients are GEMMs / column sums over those (done by the caller).
 * Pointers need only fp32 (4-byte) alignment.  n_units = 100 with a 16-byte-aligned gx selects the tensor-core
 * forward, and n_units = 100 with 16-byte-aligned stash, out and dout the tensor-core backward; every other call runs
 * the generic kernels, which compute the same recurrence. */
int isa_gru_scan_fwd(const float* gx, const float* w_hh, const float* b_hh, const float* b_ih, int n_seq, int T, int n_units,
                     int inner, long long outer_tok_stride, long long inner_tok_stride, long long t_tok_stride,
                     float* out, float* stash, isa_stream_t stream);

int isa_gru_scan_bwd(const float* dout, const float* out, const float* stash, const float* w_hh,
                     int n_seq, int T, int n_units,
                     int inner, long long outer_tok_stride, long long inner_tok_stride, long long t_tok_stride,
                     float* dgx, float* dghn, isa_stream_t stream);

/* ------------------------------------------------------------------ masked softmax over H*W
 * Replaces the masked spatial softmaxes of the live attention layers:
 *   /root/reference/code/lib/archs/modules/utils.py:507-512  SpatialAttentionLayer.forward
 *       beta.masked_fill(1 - y, -inf) -> softmax over H*W -> * sum(y)          (K = 1, scale = sum(y), NaN kept)
 *   /root/reference/code/lib/archs/modules/utils.py:648-652  HardAttentionLayer.forward
 *       e_t.expand(-1, n, ..).masked_fill(1 - ins_seg, -inf) -> softmax over H*W -> NaN -> 0   (K = n instances)
 * x     [B][HW] f32     one logit map per image, shared by its K masks
 * mask  [B][K][HW]      mask_kind 0: u8, 1: f32; non-zero = pixel takes part
 * scale [B*K] or NULL   multiplies row (b,k) of the result
 * y     [B][K][HW]      softmax restricted to the mask, 0 elsewhere; a row whose mask is empty is NaN
 *                       everywhere (what softmax over all -inf gives) or 0 everywhere with nan_to_zero
 * stats [B*K][2]        (max, sum of exponentials) per row, needed by the backward call
 * Backward: dx[b][p] = sum_k y[b][k][p] * (dy[b][k][p] - (sum_q y[b][k][q] dy[b][k][q]) / scale[b][k]);
 * rows with an empty mask contribute nothing (masked_fill's backward zeroes them). */
size_t isa_masked_softmax_hw_workspace_bytes(int B, int K, int HW);
int isa_masked_softmax_hw_fwd(const float* x, const void* mask, int mask_kind, int B, int K, int HW, const float* scale,
                              int nan_to_zero, float* y, float* stats, void* workspace, size_t workspace_bytes,
                              isa_stream_t stream);
int isa_masked_softmax_hw_bwd(const float* y, const float* dy, const float* stats, const float* scale, int B, int K, int HW,
                              float* dx, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ row reductions / row affine
 * The squeeze-excite channel attention (/root/reference/code/lib/archs/modules/utils.py:402-420 AttentionLayer):
 * global average pool = row sums over H*W, x * gate = row affine; their gradients are the same two primitives.
 *   isa_row_dot     out[r] = sum_p a[r][p] * b[r / b_rows_div][p]   (b NULL: plain row sums); deterministic two-stage
 *   isa_row_affine  y[r][p] = x[r][p] * g[r] + c[r]                 (c NULL: 0) */
size_t isa_row_dot_workspace_bytes(int rows, int HW);
int isa_row_dot(const float* a, const float* b, int rows, int HW, int b_rows_div, float* out, void* workspace,
                size_t workspace_bytes, isa_stream_t stream);
int isa_row_affine(const float* x, const float* g, const float* c, int rows, int HW, float* y, isa_stream_t stream);

/* ------------------------------------------------------------------ masked batch norm
 * /root/reference/code/lib/archs/modules/utils.py:568-591 maskBN.forward in training mode (HardAttentionLayer's
 * normalisation over the foreground, :645): mm[b] = sum of the mask over all channels and pixels + 1,
 *   mean[c] = (1/B) sum_b (sum_p x m) / mm[b],  var[c] = (1/B) sum_b (sum_p (x - mean[c])^2 m) / mm[b],
 *   y = (x - mean) / sqrt(var + eps) * weight + bias  (weight / bias NULL: 1 / 0).
 * x, y [B][C][HW] f32; mask [B][mask_channels][HW] f32 with mask_channels 1 (shared by the channels) or C.
 * stats [2*C + B*mask_channels]: mean, var (what the running averages are updated from) and the mask sums the
 * backward call needs.  Backward differentiates through mean and var like the reference's autograd graph:
 * dx [B][C][HW], dweight / dbias [C] (NULL: skipped); no gradient for the mask.  Deterministic two-stage sums. */
size_t isa_mask_bn_workspace_bytes(int B, int C, int HW);
int isa_mask_bn_fwd(const float* x, const float* mask, int mask_channels, int B, int C, int HW, const float* weight,
                    const float* bias, float eps, float* y, float* stats, void* workspace, size_t workspace_bytes,
                    isa_stream_t stream);
int isa_mask_bn_bwd(const float* x, const float* mask, int mask_channels, const float* dy, const float* stats,
                    const float* weight, float eps, int B, int C, int HW, float* dx, float* dweight, float* dbias,
                    void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ single-query readout
 * /root/reference/code/lib/archs/modules/utils.py:59-69 Decoder.forward: sigmoid(bmm(q (b,1,C), enc (b,C,HW))).
 * q [B][C], enc [B][C][HW], out [B][HW].  Backward writes dz = dout * out * (1 - out) [B][HW] and, if denc is
 * not NULL, denc[b][c][p] = q[b][c] * dz[b][p]; dq is isa_row_dot(enc, dz, B*C, HW, C). */
int isa_readout_fwd(const float* q, const float* enc, int B, int C, int HW, float* out, isa_stream_t stream);
int isa_readout_bwd(const float* q, const float* out, const float* dout, int B, int C, int HW, float* dz, float* denc,
                    isa_stream_t stream);

/* ------------------------------------------------------------------ local 3x3 dilated attention
 * /root/reference/code/lib/archs/modules/utils.py:267-303 _ScalePDAttention.forward (the stencil part between the
 * 1x1 projections and the output 1x1 convolution): per pixel, softmax over its nine dilated neighbours.
 * Q, K [Bh][dk][h][w], V [Bh][dv][h][w] f32 (heads folded into the batch as the reference's .view does);
 * nomask [mask_batches][h][w] f32 or NULL, non-zero = neighbour excluded; image b uses nomask[b % mask_batches]
 * (the reference tiles the mask with .repeat(n_head,1,1,1), utils.py:272); out-of-image neighbours are zero padding
 * that takes part with score 0 (utils.py:281-285).  out [Bh][dv][h][w]; P [Bh][9][h][w] = the probabilities, saved
 * for backward (NULL at inference).  Backward needs a [Bh][9][h][w] f32 workspace. */
int isa_local_attention_fwd(const float* Q, const float* K, const float* V, const float* nomask, int mask_batches, int Bh,
                            int dk, int dv, int h, int w, int dil, float scale, float* out, float* P, isa_stream_t stream);
int isa_local_attention_bwd(const float* Q, const float* K, const float* V, const float* P, const float* dout, int Bh,
                            int dk, int dv, int h, int w, int dil, float scale, float* dQ, float* dK, float* dV,
                            float* dS_workspace, isa_stream_t stream);

/* ------------------------------------------------------------------ channels-last epilogues, residual + LayerNorm
 * Token-major [rows][C] f32 matrices (an NHWC activation is one with rows = N*H*W).
 *   isa_bias_act_*       the `+ bias` / ReLU that follows every convolution of the embedding network
 *                        (/root/reference/code/lib/archs/modules/vgg16.py:82-140 conv+ReLU stacks, reseg.py:117-121
 *                        transposed convolutions + ReLU): y = act(x + b) in place on a bias-free convolution output;
 *                        backward gx = gy * (y > 0) and dbias = column sums of gx in one pass (deterministic).
 *   isa_add_layernorm_*  MultiHeadAttention's `self.layer_norm(output + residual)`
 *                        (/root/reference/code/lib/archs/modules/utils.py:218-219), nn.LayerNorm semantics (biased
 *                        variance, eps inside the root); backward returns the gradient of (x + res) and of gamma/beta. */
size_t isa_bias_act_workspace_bytes(int C);
int isa_bias_act_fwd(float* x, const float* bias, long long rows, int C, int relu, isa_stream_t stream);
int isa_bias_act_bwd(const float* gy, const float* y, float* gx, float* dbias, long long rows, int C, int relu, void* workspace,
                     size_t workspace_bytes, isa_stream_t stream);
size_t isa_add_layernorm_workspace_bytes(long long rows, int C);
int isa_add_layernorm_fwd(const float* x, const float* res, const float* gamma, const float* beta, long long rows, int C, float eps,
                          float* y, float* stats, isa_stream_t stream);
int isa_add_layernorm_bwd(const float* gy, const float* x, const float* res, const float* gamma, const float* stats, long long rows,
                          int C, float* gv, float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ pixel heads (1x1 convolutions -> NCHW planes)
 * /root/reference/code/lib/archs/reseg.py:122-126: the semantic and the embedding head are 1x1 convolutions over the
 * same feature map (here the channel concatenation [up-sampled features | skip], never materialised).
 *   xa [P][Ca], xb [P][Cb] f32 NHWC sources (P = n * HW pixels; xb may be NULL with Cb = 0; Ca, Cb even);
 *   w [Co0 + Co1][Ca + Cb] the two heads' weights stacked, bias [Co0 + Co1] or NULL;
 *   out0 [n][Co0][HW], out1 [n][Co1][HW] f32 NCHW planes -- what isa_disc_loss_* / isa_fg_compact read.
 * Backward writes the NHWC source gradients ga / gb (either may be NULL) from the NCHW output gradients g0 / g1 (either
 * may be NULL = zero); weight and bias gradients are plain GEMMs / row sums (host side).  Co0 + Co1 <= 32. */
int isa_pixel_heads_fwd(const float* xa, int Ca, const float* xb, int Cb, const float* w, const float* bias, float* out0, int Co0,
                        float* out1, int Co1, long long P, int HW, isa_stream_t stream);
int isa_pixel_heads_bwd(const float* g0, int Co0, const float* g1, int Co1, const float* w, float* ga, int Ca, float* gb, int Cb,
                        long long P, int HW, isa_stream_t stream);
/* dw_db = [ dw [Co0+Co1][Ca+Cb] | db [Co0+Co1] ] from the NCHW output gradients and the NHWC sources (deterministic:
 * per-CTA partials in the workspace, fixed-order final sum). */
size_t isa_pixel_heads_wgrad_workspace_bytes(int Ca, int Cb, int Co0, int Co1);
int isa_pixel_heads_wgrad(const float* g0, int Co0, const float* g1, int Co1, const float* xa, int Ca, const float* xb, int Cb,
                          long long P, int HW, float* dw_db, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ 2x2 / stride-2 max pool (NHWC)
 * The nn.MaxPool2d(2, 2) between the backbone's convolution stages (/root/reference/code/lib/archs/modules/vgg16.py:82-140)
 * on channels-last activations: x [N][H][W][C] -> y [N][H/2][W/2][C] (floor mode, C % 4 == 0); idx (u8, shape of y, NULL at
 * inference) records the window position 0..3 of the maximum (first maximum in row-major order, NaN wins, like PyTorch);
 * the backward scatters gy through idx into gx [N][H][W][C].  skip_grad (optional, NULL = none): a second gradient of x --
 * the skip connection that consumes the same activation (vgg16.py returns the stage outputs as skips) -- given as
 * [N][H][W] pixels of C floats with a pixel stride of skip_pixel_stride floats (a channel slice of a wider NHWC gradient,
 * e.g. torch.cat's backward) and added in the same pass: gx = scatter(gy) + skip_grad. */
int isa_maxpool2x2_fwd(const float* x, int N, int H, int W, int C, float* y, unsigned char* idx, isa_stream_t stream);
int isa_maxpool2x2_bwd(const float* gy, const unsigned char* idx, int N, int H, int W, int C, const float* skip_grad,
                       long long skip_pixel_stride, float* gx, isa_stream_t stream);

/* ------------------------------------------------------------------ instance-count tail (ReSeg(count_head=True))
 * The end of the count branch: conv4's bias + ReLU epilogue, global average pool, the 64 -> 1 linear layer, sigmoid,
 * count-regression loss and rounding, as one forward and one streaming backward.  The branch is this project's own
 * specification (archs.py); its float64 restatement is oracle/count_head_ref.py.
 *   x          [bs][P][C] f32 NHWC: the bias-free conv4 output, finished IN PLACE to y = relu(x + conv_bias) (kept for
 *              the backward); conv_bias [C], w [C] (the linear layer's weight row), b [1]
 *   pooled     [bs][C] = mean_p y;  s [bs] = sigmoid(pooled . w + b);  n_pred [bs] i32 = clamp(rint(s * K), 1, K)
 *              (round half to even, like torch.round)
 *   n_objects  [bs] i32, or NULL (inference: then loss must be NULL too)
 *   loss       [1] = mean_b (s_b - n_objects_b / K)^2, or NULL
 * Backward, with dz_b = grad_loss * 2 (s_b - n_objects_b / K) / bs * s_b (1 - s_b):
 *   gx [bs][P][C] = (y > 0) dz_b w_c / P;  dconv_bias [C] = sum_{b,p} gx;  dw [C] = sum_b dz_b pooled[b];  db [1] = sum_b dz_b.
 * workspace  isa_count_head_workspace_bytes(bs, P, C) bytes; hand the SAME buffer, untouched, to the backward (it
 *            carries the forward's per-(b, c) counts of y > 0, so the bias gradient needs no pass over the map).
 * Limits: 1 <= bs <= 65535, 1 <= P, C % 4 == 0 and 4 <= C <= 256, 1 <= K <= 254; x, conv_bias, y, gx, w 16-byte
 * aligned.  A rejected call enqueues nothing.  Deterministic: fixed-order sums, no float atomics. */
size_t isa_count_head_workspace_bytes(int bs, long long P, int C);
int isa_count_head_fwd(float* x, const float* conv_bias, const float* w, const float* b, const int* n_objects,
                       int bs, long long P, int C, int K, float* pooled, float* s, int* n_pred, float* loss,
                       void* workspace, size_t workspace_bytes, isa_stream_t stream);
int isa_count_head_bwd(const float* y, const float* pooled, const float* s, const float* w, const int* n_objects,
                       const float* grad_loss, int bs, long long P, int C, int K,
                       float* gx, float* dconv_bias, float* dw, float* db,
                       void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ training-set augmentation (isa_b200.augment)
 * Gathers a batch of augmented training samples from a device-resident store of decoded images.  The geometry (which
 * maps are drawn) is the host's; this call applies them.  Its numpy restatement is oracle/augment_ref.py.
 *   rgb        [sum h*w][3] u8 and labels [sum h*w] u8 (ids 0..n-1, 255 = background): the images, packed
 *   store      [n_images][3] i64 = (pixel offset, h, w) of each image; 1 <= h, w <= 32767, offset + h*w <= store_pixels
 *   params     [b][7] i64 = (source image index, a0..a5): the inverse map output -> source in Q32.32 fixed point,
 *              |a_i| < 2^44.  Output pixel (x, y) reads the source at, exactly in int64 and in units of 2^-33,
 *                u = a0 (2x+1) + a1 (2y+1) + 2 a2,   v = a3 (2x+1) + a4 (2y+1) + 2 a5
 *              label = nearest pixel (u >> 33, v >> 33), 255 outside the source; rgb = bilinear from the four taps
 *              around (u - 2^32, v - 2^32), taps outside the source read 0, fp32 weights from the low 33 bits.
 *   h_mean_std [6] f32 on the HOST: mean[3], std[3];  image = (rgb / 255 - mean) / std
 * Outputs, in the layouts Model.train_step reads:
 *   image [b][H][W][3] f32 (a (b,3,H,W) tensor in channels_last), sem [b][H][W] u8 = (ins != 255),
 *   ins [b][H][W] u8, n_objects [b] i32.
 * The ids present in a sample are renumbered 0..n-1 in ascending order of the source id (nearest sampling, rotation
 * and cutting drop instances); n_objects = n.  A sample left with no instance is rendered again through the plain
 * resize map (a0 = round(w 2^32 / W), a4 = round(h 2^32 / H), the rest 0), so n_objects is 0 only if that view has
 * no instance either.  A map that breaks the limit above counts as a view with no instance, so the sample gets the
 * plain view; a sample whose source index or store entry is invalid is written black and empty (n_objects 0).
 * Integer atomics only: the same call writes the same bytes.
 * workspace  isa_augment_workspace_bytes(b) bytes, 4-byte aligned.
 * Limits: 1 <= b <= 65535, 1 <= H, W <= 32767, std non-zero (else ISA_ERR_BAD_ARG; a rejected call
 * enqueues nothing). */
size_t isa_augment_workspace_bytes(int b);
int isa_augment(const unsigned char* rgb, const unsigned char* labels, const long long* store, int n_images,
                long long store_pixels, const long long* params, int b, int H, int W, const float* h_mean_std,
                float* image, unsigned char* sem, unsigned char* ins, int* n_objects,
                void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ fused gradient clipping + Adadelta
 * The tail of the reference's training step (/root/reference/code/lib/model.py:271-281: clip_grad_norm_ then
 * optimizer.step(); settings/CVPPP/training_settings.py: OPTIMIZER 'Adadelta', LEARNING_RATE 1, WEIGHT_DECAY 1e-3,
 * CLIP_GRAD_NORM 10) over flat fp32 buffers.  PyTorch's Adadelta arithmetic:
 *   g += wd p;  v = rho v + (1-rho) g^2;  d = sqrt(u + eps) / sqrt(v + eps) g;  u = rho u + (1-rho) d^2;  p -= lr d */
size_t isa_adadelta_workspace_bytes(void);
int isa_adadelta_step(float* param, const float* grad, float* square_avg, float* acc_delta, long long n, float lr, float rho, float eps,
                      float weight_decay, float max_norm, float* norm_out, void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ fused semantic-head losses (cross entropy + Dice)
 * Replaces, on the training step,
 *   /root/reference/code/lib/losses/dice.py:10-51 (dice_coefficient), :54-89 (dice_loss, mean reduction) and the
 *   CrossEntropyLoss(class_weights) call of /root/reference/code/lib/model.py:255-263
 * with one forward and one backward pass over the logits.
 * logits        [bs][n_classes][HW] f32 (NCHW planes), 2 <= n_classes <= 8
 * class_map     [bs][HW] u8 class index per pixel (isa_onehot_argmax distils the collate's one-hot once)
 * class_weights [n_classes] f32 or NULL (the same vector weights both losses, model.py:113-127)
 * dice_time     1: den = sum p + sum t (what Model passes, model.py:264);  2: sum p^2 + sum t^2
 * out_ce_dice   [2] f32: weighted-mean cross entropy, mean Dice loss (background dropped unless optimize_bg)
 * workspace     isa_seg_losses_workspace_bytes bytes; hand the SAME buffer to isa_seg_losses_bwd.
 * Deterministic (fixed-order partial sums, no float atomics). */
size_t isa_seg_losses_workspace_bytes(int bs, int n_classes, long long HW);
int isa_seg_losses_fwd(const float* logits, const unsigned char* class_map, const float* class_weights,
                       int bs, int n_classes, long long HW, int dice_time, float smooth, int optimize_bg,
                       float* out_ce_dice, void* workspace, size_t workspace_bytes, isa_stream_t stream);
/* grad_ce / grad_dice: device scalars (NULL = 0); grad_logits [bs][n_classes][HW] out. */
int isa_seg_losses_bwd(const float* logits, const unsigned char* class_map, const float* class_weights,
                       int bs, int n_classes, long long HW, int dice_time, const float* grad_ce,
                       const float* grad_dice, float* grad_logits, const void* workspace, size_t workspace_bytes,
                       isa_stream_t stream);
/* Dense one-hot [bs][n_classes][HW] (target_kind 1 f32, 2 i64, 3 u8) -> u8 class map, first maximum wins
 * (Tensor.max(1)[1], model.py:256-257). */
int isa_onehot_argmax(const void* target, int target_kind, int bs, int n_classes, long long HW,
                      unsigned char* class_map, isa_stream_t stream);

/* ------------------------------------------------------------------ ReNet projection GEMMs (tcgen05, fused bf16 hi/lo split)
 * The GEMMs around the GRU scan of the ReNet contract (/root/reference/code/lib/archs/modules/README.md:225-256; nn.GRU's
 * x W_ih^T and autograd's dG W_ih, dG^T [x | h_prev | 1]).  fp32 operands are read ONCE from global memory and split into
 * bf16 hi + lo parts inside the kernel (a b ~= a_hi b_hi + a_hi b_lo + a_lo b_hi, fp32 accumulation in tensor memory,
 * error ~2^-16 relative); nothing is transposed, concatenated or copied.  All widths multiples of 4, pointers 16 B aligned.
 *   fwd    gx [tokens][n_out] = x [tokens][cin] w [n_out][cin]^T          (n_out = 2 directions x 3 gates x n)
 *   dx     dx [tokens][cin]   = dg [tokens][n_out] w [n_out][cin]
 *   wgrad  dw_ih [2][3n][cin], dw_hh [2][3n][n], db_ih [2][3n], db_hh [2][3n] from dgx [tokens][2][3n], dghn [tokens][2][n],
 *          x [tokens][cin] and the forward output out [tokens][2][n]: h_{t-1} of direction 0 is out's row `step` tokens back,
 *          of direction 1 `step` tokens ahead, zero outside the sweep (position = (token / pos_div) % pos_mod).  The token
 *          dimension is split over CTAs and the partials are folded in a fixed order (deterministic). */
/* fwd / dx: the (small, L2-resident) weight operand is packed once per call into the kernel's shared-memory tile images in
 * `workspace` (isa_renet_proj_workspace_bytes(cin, n_out) bytes) and streamed by bulk copies; the token operand is split on the fly. */
size_t isa_renet_proj_workspace_bytes(int cin, int n_out);
int isa_renet_proj_fwd(const float* x, const float* w, long long tokens, int cin, int n_out, float* gx, void* workspace,
                       size_t workspace_bytes, isa_stream_t stream);
int isa_renet_proj_dx(const float* dg, const float* w, long long tokens, int n_out, int cin, float* dx, void* workspace,
                      size_t workspace_bytes, isa_stream_t stream);
size_t isa_renet_proj_wgrad_workspace_bytes(long long tokens, int cin, int n);
int isa_renet_proj_wgrad(const float* dgx, const float* dghn, const float* x, const float* out, long long tokens, int cin, int n,
                         long long step, int pos_div, int pos_mod, float* dw_ih, float* dw_hh, float* db_ih, float* db_hh,
                         void* workspace, size_t workspace_bytes, isa_stream_t stream);

/* ------------------------------------------------------------------ SBD / |DiC| of instance label images
 * Replaces the numpy loops of /root/reference/code/evaluate.py:18-57 (calc_dice, calc_bd, calc_sbd, calc_dic):
 * gt, pred [n_images][pixels_per_image] u8 label images (0 = background) ->
 * out [n_images][5] f64 = {SBD, BD(gt, pred), BD(pred, gt), #objects(gt), #objects(pred)}; |DiC| = |out[3] - out[4]|.
 * One contingency-table pass (integer atomics, exact) + a per-image reduction; every dice is the reference's ratio of
 * integer counts in float64.  NaN where the reference returns nan (no object in the first image) or raises (none in the
 * second).  workspace: isa_sbd_workspace_bytes(n_images). */
size_t isa_sbd_workspace_bytes(int n_images);
int isa_sbd(const unsigned char* gt, const unsigned char* pred, int n_images, long long pixels_per_image, double* out,
            void* workspace, size_t workspace_bytes, isa_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ISA_B200_H_ */
