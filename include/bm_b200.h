/* brainmagick_b200 -- C ABI of the B200-native contrastive training step (SimpleConv + ClipLoss).
 *
 * The reference (facebookresearch/brainmagick) has no FFI: its boundary for this path is the Python object
 * surface of `bm.models.SimpleConv` (bm/models/simpleconv.py:22-249) and `bm.losses.ClipLoss`
 * (bm/losses.py:29-114), called from bm/solver.py:297,373 and bm/train.py:84-86.  The drop-in modules in
 * `brainmagick_b200/` keep that surface and call THIS library through ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is DEVICE memory unless stated; fp32 data, int32 indices,
 *     fp64 only for the small statistics scratch buffers;
 *   - the caller owns every buffer (inputs, outputs, saved activations, scratch); the library never allocates;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no entry point synchronises;
 *   - returns 0 on success, non-zero on error; `bm_last_error()` gives the message (thread local);
 *   - activations inside the encoder are channels-last [B, T, C]; the model input `meg` [B, C, T], the encoder
 *     output `estimate` [B, F, T] and the `candidates` [B', F, T] keep the reference's channel-major layout.
 * There is no CPU fallback anywhere in this library.
 */
#ifndef BM_B200_H_
#define BM_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef void* bm_stream_t;

const char* bm_last_error(void);
int bm_abi_version(void);
/* number of CUDA kernels this library has launched since it was loaded (bench.py's `gpu_launches`). */
unsigned long long bm_launch_count(void);
/* experiment switches (returns the previous value).  By default bm_tc_wgrad keeps X raw in shared memory as the tf32
 * `hi` operand (the tensor core ignores the 13 low mantissa bits) and only writes `lo = x - trunc(x)`; bit 0 restores
 * the explicit round-to-nearest hi/lo split (one third more shared-memory traffic). */
int bm_set_debug_flags(int flags);
/* profiling aid (process-wide, NOT part of the product path): device buffer of >= 8 * gridDim long longs that the CTA-pair
 * weight-gradient kernel fills with per-CTA cycle counters (barrier waits per warp role); NULL (default) disables it. */
int bm_set_debug_buffer(long long* buf);

/* ---- K1: spatial-attention weights, once per recording ------------------------------------------------
 * replaces FourierEmb.forward (bm/models/common.py:254-271) + the score/softmax half of ChannelMerger.forward
 * (common.py:337-357).  positions [R,C,2] (INVALID=-0.1 marks padded sensors), freq [n] = 2*pi*arange(n)/1.4
 * with n = sqrt(P/2), heads [O,P], ban_centre [2] or NULL (eval / dropout 0).
 * out: emb [R,C,P] (saved for backward), weights [R,O,C] = softmax over C. */
int bm_attention_weights_fwd(const float* positions, const float* freq, const float* heads,
                             const float* ban_centre, float radius, int R, int C, int O, int P, float* emb,
                             float* weights, bm_stream_t stream);
/* dweights [R,O,C] -> dheads [O,P]; dscores is [R,O,C] scratch. */
int bm_attention_weights_bwd(const float* dweights, const float* weights, const float* emb, int R, int C, int O,
                             int P, float* dscores, float* dheads, bm_stream_t stream);

/* K1 in pieces (the two contractions -- scores = emb heads^T and dheads = dscores^T emb -- then run on the tensor-core
 * kernels bm_tc_conv1d_persistent(out_tmajor) / bm_tc_wgrad): Fourier embedding, in-place masked softmax, softmax backward. */
int bm_fourier_emb(const float* positions, const float* freq, int R, int C, int P, float* emb, bm_stream_t stream);
int bm_masked_softmax(float* weights, const float* positions, const float* ban_centre, float radius, int R, int O, int C,
                      bm_stream_t stream);
int bm_softmax_bwd(const float* weights, const float* dweights, long long rows, int C, float* dscores,
                   bm_stream_t stream);

/* ---- K2: sensor chain ----------------------------------------------------------------------------------
 * replaces the mixing einsum of ChannelMerger.forward (common.py:358), `initial_linear` (simpleconv.py:113-120,
 * 213-214) and SubjectLayers.forward (common.py:55-58):
 *   u[b,t,o] = sum_c weights[rec[b],o,c] meg[b,c,t];  v = il_w u + il_b;  x0[b,t,d] = sum_p subj_w[subj[b],p,d] v[b,t,p]
 * meg [B,C,T]; il_w [IL,O]; subj_w [S,IL,D]; out u [B,T,O], v [B,T,IL], x0 [B,T,ld_x0] (channels-last; ld_x0 >= D
 * lets the caller keep x0 zero-padded to a multiple of 32 channels for the tensor-core conv that follows). */
int bm_sensor_chain_fwd(const float* meg, const float* weights, const int* rec_of_sample, const float* il_w,
                        const float* il_b, const float* subj_w, const int* subject, int B, int C, int T, int O,
                        int IL, int D, int ld_x0, float* u, float* v, float* x0, bm_stream_t stream);
/* dx0 [B,T,D] -> d_subj_w [S,IL,D], d_il_w [IL,O], d_il_b [IL], d_weights [R,O,C].
 * (subj_order, subj_off[S+1]) and (rec_order, rec_off[R+1]) are CSR groupings of the samples by subject and by
 * recording; dv [B,T,IL] and du [B,T,O] are scratch. */
int bm_sensor_chain_bwd(const float* dx0, const float* meg, const float* il_w, const float* subj_w,
                        const int* subject, const float* u, const float* v, const int* subj_order,
                        const int* subj_off, const int* rec_order, const int* rec_off, int B, int C, int T, int O,
                        int IL, int D, int ld_x0, int S, int R, float* dv, float* du, float* d_subj_w, float* d_il_w,
                        float* d_il_b, float* d_weights, bm_stream_t stream);

/* The same chain as separate stages with explicit leading dimensions (u / v / dv / du / x0 may be kept zero-padded to a
 * multiple of 64 channels so that `initial_linear` runs on the tensor-core pointwise kernel, bm_tc_conv1d_persistent Kw=1). */
int bm_sensor_mix_fwd(const float* meg, const float* weights, const int* rec_of_sample, int B, int C, int T, int O,
                      int ld_u, float* u, bm_stream_t stream);
int bm_initial_linear_fwd(const float* u, int ld_u, const float* il_w, const float* il_b, int B, int T, int O, int IL,
                          int ld_v, float* v, bm_stream_t stream);
int bm_subject_layers_fwd(const float* v, int ld_v, const float* subj_w, const int* subject, int B, int T, int IL, int D,
                          int ld_x0, float* x0, bm_stream_t stream);
int bm_subject_layers_bwd(const float* dx0, int ld_x0, const float* v, int ld_v, const float* subj_w, const int* subject,
                          const int* subj_order, const int* subj_off, int B, int T, int IL, int D, int S, int ld_dv,
                          float* dv, float* d_subj_w, bm_stream_t stream);
int bm_initial_linear_bwd(const float* dv, int ld_dv, const float* u, int ld_u, const float* il_w, int B, int T, int O,
                          int IL, int ld_du, float* du, float* d_il_w, float* d_il_b, bm_stream_t stream);
int bm_sensor_mix_bwd(const float* du, int ld_du, const float* meg, const int* rec_order, const int* rec_off, int B, int C,
                      int T, int O, int R, float* d_weights, bm_stream_t stream);

/* ---- K3: dilated Conv1d + train-mode BatchNorm + GELU + skip (ConvSequence, common.py:98-151) ------------
 * w [Cout,Cin,Kw] -> wf [Kw,Cin,Cout] (forward operand), wb [Kw,Cout,Cin] (data-gradient operand). */
int bm_conv_weight_prep(const float* w, int Cout, int Cin, int Kw, float* wf, float* wb, bm_stream_t stream);
/* y[b,t,o] = bias[o] + sum_{i,j} w[o,i,j] x[b, t+(j-Kw/2)*dilation, i]  (zero outside [0,T)); x,y channels-last.
 * stats (nullable): fp64 [2*Cout] receiving sum(y), sum(y^2) over (b,t) -- zeroed by this call. */
int bm_conv1d_fwd(const float* x, const float* wf, const float* bias, int B, int T, int Cin, int Cout, int Kw,
                  int dilation, float* y, double* stats, bm_stream_t stream);
/* batch statistics -> mean, invstd; updates running stats (nullable) like nn.BatchNorm1d(momentum). */
int bm_bn_stats_finalize(const double* stats, long long n, float eps, float momentum, float* running_mean,
                         float* running_var, float* mean, float* invstd, int C, bm_stream_t stream);
int bm_bn_eval_stats(const float* running_mean, const float* running_var, float eps, float* mean, float* invstd,
                     int C, bm_stream_t stream);
/* x_new = GELU(gamma*(y-mean)*invstd + beta) (+ x_old if not NULL); rows = B*T.
 * amax_out (nullable; the same argument on bm_bn_gelu_skip_bwd, bm_glu_bwd, bm_tc_conv1d_f16): a device float that receives
 * max |output| -- the x_amax of the F16-pipe conv (bm_tc_conv1d_f16) that consumes the tensor next, produced by the kernel
 * that writes the tensor instead of a separate bm_amax pass over it. */
int bm_bn_gelu_skip_fwd(const float* y, const float* mean, const float* invstd, const float* gamma,
                        const float* beta, const float* x_old, float* x_new, long long rows, int C, float* amax_out,
                        bm_stream_t stream);
/* g = dL/dx_new -> dy (through GELU and BN), dgamma, dbeta.  batch_stats=1: training-mode BN backward.
 * sums: fp64 [2*C] scratch. */
int bm_bn_gelu_skip_bwd(const float* g, const float* y, const float* mean, const float* invstd,
                        const float* gamma, const float* beta, int batch_stats, long long rows, int C,
                        double* sums, float* dy, float* dgamma, float* dbeta, float* amax_out /* of dy */,
                        bm_stream_t stream);
/* dx = conv_transpose(dy) (+ addend, the skip-path gradient, if not NULL). */
int bm_conv1d_bwd_data(const float* dy, const float* wb, const float* addend, int B, int T, int Cin, int Cout,
                       int Kw, int dilation, float* dx, bm_stream_t stream);
/* dw [Cout,Cin,Kw] (reference layout), dbias [Cout]. */
int bm_conv1d_bwd_weight(const float* dy, const float* x, int B, int T, int Cin, int Cout, int Kw, int dilation,
                         float* dw, float* dbias, bm_stream_t stream);

/* ---- K4: Conv1d(H -> 2H, Kw, pad=Kw/2) + GLU (common.py:133-138) ----------------------------------------
 * wf [Kw,Cin,2H]; h (nullable, saved for backward) [B,T,2H]; out [B,T,H] = h[:, :H] * sigmoid(h[:, H:]). */
int bm_conv1d_glu_fwd(const float* x, const float* wf, const float* bias, int B, int T, int Cin, int H, int Kw,
                      float* h, float* out, bm_stream_t stream);
int bm_glu_bwd(const float* g, const float* h, long long rows, int H, float* dh,
               float* dbias /* nullable [2H]: sum over rows of dh = the GLU conv's bias gradient, from the same pass */,
               float* amax_out /* of dh */, bm_stream_t stream);

/* ---- K5: head Conv1d(H,2H,1) -> GELU -> ConvTranspose1d(2H,F,1) (simpleconv.py:185-189,246-249) --------
 * x [B,T,H]; w0 [2H,H]; w2 [2H,F] (ConvTranspose1d weight is input-major); out h1,q [B,T,2H], est [B,F,T]. */
int bm_head_fwd(const float* x, const float* w0, const float* b0, const float* w2, const float* b2, int B, int T,
                int H, int F, float* h1, float* q, float* est, bm_stream_t stream);
/* dest [B,F,T] -> dx [B,T,H], dw0 [2H,H], db0 [2H], dw2 [2H,F], db2 [F]; dq [B,T,2H] scratch. */
int bm_head_bwd(const float* dest, const float* x, const float* w0, const float* w2, const float* h1,
                const float* q, int B, int T, int H, int F, float* dq, float* dx, float* dw0, float* db0,
                float* dw2, float* db2, bm_stream_t stream);

/* parameter-gradient half of bm_head_bwd, for callers that compute dq and dx themselves (tensor-core path):
 * in: dq = d(loss)/dq [B,T,2H]; out: dw2, db2, dq <- dq*GELU'(h1) (in place), dw0, db0. */
int bm_head_bwd_params(const float* dest, const float* x, const float* h1, const float* q, int B, int T, int H, int F,
                       float* dq, float* dw0, float* db0, float* dw2, float* db2, bm_stream_t stream);

/* ---- K6: ClipLoss (bm/losses.py:77-114) -----------------------------------------------------------------
 * est [Bn,KT], cand [Bc,KT] (KT = F*T, any consistent flattening).
 * bm_clip_scores = ClipLoss.get_scores (+ get_probabilities when probs != NULL):
 *   inv_norm[o] = 1/(1e-8+||cand_o||), scores[b,o] = inv_norm[o] <est_b, cand_o>, probs = softmax_o(scores).
 *   norms_given = 1: inv_norm is an INPUT (a fixed candidate set is normed once, see bm_candidate_inv_norms).
 * One split-K tcgen05 GEMM on CTA pairs (3xTF32; every accumulation chain is bounded to 64 K-steps and drained into an
 * fp32 round-to-nearest running sum, because the tensor core's accumulator truncates) that also produces the candidate
 * norms, + one finalize kernel (slice reduction in a fixed order, norm scale, row softmax / cross-entropy / batch mean).
 * workspace: bm_clip_workspace(Bn,Bc,KT) floats of caller-owned scratch, 8-byte aligned; status: device int set on a
 * pipeline timeout (never hangs).  KT % 4 != 0 (no TMA row pitch) falls to the FP32-FMA GEMM of this library. */
long long bm_clip_workspace(int Bn, int Bc, long long KT);
int bm_clip_scores(const float* est, const float* cand, int Bn, int Bc, long long KT, int norms_given, float* inv_norm,
                   float* scores, float* probs, float* workspace, long long workspace_floats, int* status,
                   bm_stream_t stream);
/* inv_norm[o] = 1/(1e-8+||cand_o||) alone (losses.py:91); ss fp64 [Bc] scratch. */
int bm_candidate_inv_norms(const float* cand, int Bc, long long KT, double* ss, float* inv_norm, bm_stream_t stream);
/* ClipLoss.forward: loss = mean_b CE(scores[b,:], target_offset + b).  target_offset = 0 is the reference;
 * rank*Bn is the multi-GPU extension with all-gathered candidates.  row_loss [Bn], loss [1]; inv_norm, scores, probs
 * are outputs kept for the backward. */
int bm_clip_loss_fwd(const float* est, const float* cand, int Bn, int Bc, long long KT, int target_offset,
                     float* inv_norm, float* scores, float* probs, float* row_loss, float* loss, float* workspace,
                     long long workspace_floats, int* status, bm_stream_t stream);
/* dL/dest [Bn,KT] = gout * ((probs - onehot)/Bn * inv_norm) @ cand ; G [Bn,Bc] scratch; gout [1] on device. */
int bm_clip_loss_bwd(const float* probs, const float* inv_norm, const float* cand, const float* gout, int Bn,
                     int Bc, long long KT, int target_offset, float* G, float* dest, int* status, bm_stream_t stream);

/* ---- Stand-alone ConvSequence / DeepMel (SURVEY 8(f) row 3): bm/models/common.py:79-151, bm/models/features.py:15-35 --
 * Layer epilogue x_new = act(bn(y)) (+ x_old) over channels-last rows [rows, C] and its backward, for the cases the
 * brain encoder's fused BatchNorm+GELU kernels do not cover: act 0 = GELU, 1 = LeakyReLU(slope) (common.py:95),
 * 2 = none; mean == NULL = no BatchNorm (the layer then only applies the activation / the skip).
 * bm_bn_act_skip_bwd: dy = d/dy of the above given g = dL/dx_new (the skip branch's gradient is g itself);
 * batch_stats=1: training-mode BatchNorm (dgamma, dbeta, fp64 sums [2C] scratch), 0: eval statistics. */
int bm_bn_act_skip_fwd(const float* y, const float* mean, const float* invstd, const float* gamma, const float* beta,
                       const float* x_old, float* x_new, long long rows, int C, int act, float slope,
                       bm_stream_t stream);
int bm_bn_act_skip_bwd(const float* g, const float* y, const float* mean, const float* invstd, const float* gamma,
                       const float* beta, int batch_stats, long long rows, int C, int act, float slope, double* sums,
                       float* dy, float* dgamma, float* dbeta, bm_stream_t stream);
/* Gradient of ClipLoss.forward w.r.t. the CANDIDATES (a trainable feature model, solver.py:304-320): with G as in
 * bm_clip_loss_bwd, dcand[o] = sum_b G[b,o] est[b] - coef[o] cand[o], coef[o] = (sum_b G[b,o] scores[b,o]) / ||cand_o||
 * (the derivative of the 1/(1e-8+||.||) normalisation, losses.py:91).  G [Bn,Bc], coef [Bc]: scratch. */
int bm_clip_loss_bwd_cand(const float* probs, const float* scores, const float* inv_norm, const float* est,
                          const float* cand, const float* gout, int Bn, int Bc, long long KT, int target_offset,
                          float* G, float* coef, float* dcand, int* status, bm_stream_t stream);

/* ---- Retrieval evaluation (SURVEY 8(f) row 1): scripts/run_eval_probs.py:237-307, bm/wer.py:80-116 ---------
 * The score matrix comes from bm_clip_scores (queries x candidates, candidate axis optionally zero-padded to the
 * tensor-core tile: ld >= n_cols); these entry points replace the host-side softmax / topk / scatter_add / label
 * comparison the reference runs per query (wer.py) or per query batch on the CPU copy (run_eval_probs.py).
 * bm_retrieval_topk, one row b of `vals` (stride ld) at a time:
 *   is_prob=0: vals are scores, p = softmax over the n_cols columns (row_max/row_sum, nullable, receive its stats);
 *   is_prob=1: vals are probabilities already, negative entries are holes;
 *   own_values [Bn] (nullable): per-row value standing in column own_col -- wer.py:93 overwrites the last negative
 *     with the query's own true output; own_labels [Bn] likewise for that column's label (wer.py:94);
 *   top_idx/top_prob [Bn,k] (nullable): the k best columns, best first, ties -> lower column (-1 / 0 if fewer);
 *   hit[b] = rank (0 = best) of the first of the k selected columns whose label is targets[b], -1 if none: a top-k'
 *     hit for any k' <= k is 0 <= hit[b] < k' (run_eval_probs.py:253-259, wer.py:107-111);
 *   soft[b] = sum of p over the columns whose label is targets[b] (wer.py:114-115).
 * bm_retrieval_probs: probs [Bn,n_cols] = softmax(scores[:, :n_cols])  (ClipLoss.get_probabilities, losses.py:97-102).
 * bm_retrieval_vocab_probs: per-word probabilities (wer.py:101-104) without atomics: vocab [Bn,V+1],
 *   vocab[b][w] = sum_{j in seg[w]..seg[w+1]} p[b][perm[j]] (+ the own candidate's p when own_word[b] == w);
 *   column V = own p when own_word[b] == V (a word no shared negative carries), else -1 (a hole for bm_retrieval_topk).
 * bm_rowdot_scaled: own[b] = <a_b, c_b> / (1e-8 + ||c_b||): the score of a query against its own true output. */
int bm_retrieval_topk(const float* vals, long long ld, int Bn, int n_cols, const float* own_values, int own_col,
                      int is_prob, int k, const long long* labels, const long long* own_labels,
                      const long long* targets, long long* top_idx, float* top_prob, int* hit, float* soft,
                      float* row_max, float* row_sum, bm_stream_t stream);
int bm_retrieval_probs(const float* scores, long long ld, int Bn, int n_cols, float* probs, bm_stream_t stream);
int bm_retrieval_vocab_probs(const float* scores, long long ld, int Bn, const float* own_scores, const float* row_max,
                             const float* row_sum, const int* perm, const int* seg, int V, const int* own_word,
                             float* vocab, bm_stream_t stream);
int bm_rowdot_scaled(const float* a, const float* c, int Bn, long long K, float* own, bm_stream_t stream);

/* ---- Batch preparation (SURVEY 8(f) row 2): bm/norm.py:239-275, 325-341; bm/solver.py:262-274 ---------------
 * bm_scale_clamp_crop: y [B,C,T_out] = op(x [B,C,T])[..., t0:t0+T_out] with op = (x - center[slot[b]][c]) / scale[..]
 *   (BatchScaler.transform; inverse=1: x*scale + center), then clamp to +-limit when clip (ScaleReject, norm.py:332-333)
 *   -- one pass, bit-identical to the reference's fp32 arithmetic.  center/scale: [R,C] tables (RobustScaler per
 *   recording, or one row of per-channel StandardScaler constants with slot = NULL).  peak_bits [B] (nullable): bit
 *   pattern of max |op(x)| over the whole uncropped sample (what ScaleReject tests, norm.py:334).
 * bm_reject_compact: keep[b] = !(peak > limit) && (mask == NULL || any(mask[b])) (norm.py:335-339);
 *   keep_rows = kept sample indices in order, n_keep[0] their count.
 * bm_gather_rows: y[i] = x[rows[i]] over rows of row_elems floats (batch[keep], norm.py:340). */
int bm_scale_clamp_crop(const float* x, const int* slot, const float* center, const float* scale, int B, int C, int T,
                        int t0, int T_out, float limit, int clip, int inverse, float* y, unsigned int* peak_bits,
                        bm_stream_t stream);
int bm_reject_compact(const unsigned int* peak_bits, const unsigned char* mask, long long mask_elems, float limit,
                      int B, unsigned char* keep, int* keep_rows, int* n_keep, bm_stream_t stream);
int bm_gather_rows(const float* x, const int* rows, int n_rows, long long row_elems, float* y, bm_stream_t stream);

/* ---- Regression objectives: L1Loss / L2Loss (bm/losses.py:11-26), the solver's 'l1' and 'mse' (bm/solver.py:76-94) -----
 * loss = mean over the selected elements of |est - out|^p (p = 1 or 2), selected = mask.expand_as(est):
 * est, out [B,F,T] fp32; mask [B,Fm,T] bytes (torch.bool: 0 / 1), Fm = 1 (one mask per sample and time, broadcast over F)
 * or Fm = F.  Unselected elements are never used arithmetically (a NaN or inf there does not reach the loss or the
 * gradient); an empty selection gives loss NaN (0/0) and zero gradients.
 * workspace: BM_REGRESSION_WS_DOUBLES doubles of caller-owned scratch.  bm_regression_loss_fwd fills it with fp64 partial
 * sums (reduced in a fixed order by the last block: the loss is bit-identical from call to call) and the selected count,
 * which bm_regression_loss_bwd reads on the device, so keep the buffer unchanged until the backward.  loss [1] fp32.
 * bm_regression_loss_bwd: dest = selected ? p |d|^(p-1) sign(d) gout / count : 0 with d = est - out (sign(0) = 0, NaN
 * propagates); dout = -dest.  gout [1] is the incoming gradient on the device; dest or dout may be NULL (not both). */
#define BM_REGRESSION_WS_DOUBLES 1186
int bm_regression_loss_fwd(const float* est, const float* out, const unsigned char* mask, int B, int F, int Fm, int T,
                           int p, double* workspace, float* loss, bm_stream_t stream);
int bm_regression_loss_bwd(const float* est, const float* out, const unsigned char* mask, const float* gout,
                           const double* workspace, int B, int F, int Fm, int T, int p, float* dest, float* dout,
                           bm_stream_t stream);

/* ---- tcgen05 (5th-gen tensor core) versions of K3/K4: 3xTF32 implicit-GEMM conv ---------------------------
 * Same arithmetic contract as bm_conv1d_fwd / bm_conv1d_bwd_data / bm_conv1d_glu_fwd (fp32-faithful: every
 * product is hi*hi + lo*hi + hi*lo of tf32 splits, fp32 accumulation in tensor memory).
 * bm_tc_weight_split: w [Cout,Cin,Kw] -> forward operand f_hi/f_lo [Kw,Cout,Cin] and data-gradient operand
 * g_hi/g_lo [Kw,Cin,Cout] (either pair may be NULL).
 * bm_tc_conv1d: x [B,T,Cin], w_hi/w_lo [Kw,Ntot,Cin]; sign=+1 forward taps, -1 data gradient; glu=1: Ntot = 2H,
 * y (nullable) receives h, glu_out [B,T,H].  status: device int (nullable) set non-zero if the kernel's pipeline
 * timed out (never hangs).  bm_tc_conv_supported: shape gate (Cin % 32, Ntot % 160 or H % 80). */
int bm_tc_conv_supported(int T, int Cin, int Ntot, int Kw, int glu);
int bm_tc_weight_split(const float* w, int Cout, int Cin, int Kw, float* f_hi, float* f_lo, float* g_hi,
                       float* g_lo, bm_stream_t stream);
int bm_tc_conv1d(const float* x, const float* w_hi, const float* w_lo, const float* bias, const float* addend,
                 int B, int T, int Cin, int Ntot, int Kw, int dilation, int sign, int glu, int act, int out_tmajor,
                 float* y, float* aux, float* glu_out, double* stats /* must be NULL: see bm_tc_conv1d_persistent */,
                 int* status, bm_stream_t stream);
/* act=1: y = GELU(.) and aux (nullable) receives the pre-activation; out_tmajor=1: y is [B,Ntot,T] (the head's
 * channel-major `estimate`).  With Kw=1 this is the pointwise (1x1) contraction of the head (K5).
 * bm_col_stats: stats[0:C] = sum_r y[r,c], stats[C:2C] = sum_r y[r,c]^2 (fp64), the BatchNorm batch statistics. */
int bm_col_stats(const float* y, long long rows, int C, double* stats, bm_stream_t stream);
/* PERSISTENT CTA-pair kernel (csrc/tc_convp.cuh): one CTA pair per SM pair loops over 256-row tiles of the flattened
 * rows b*T + t (taps that would cross a sample edge read zeros = the conv padding), epilogue warps drain tile i while the
 * operands of tile i+1 are staged.  w_raw: RAW fp32 weights re-laid K-major [Kw][Ntot][Cin] (bm_tc_weight_split with
 * f_lo / g_lo = NULL) -- the tensor core's truncation of the raw operand is the tf32 `hi`, the kernel derives `lo`.
 * accumulate=1: y += conv(x) in place (the skip-path gradient; TMA reduce-add).  glu / act / out_tmajor / aux / glu_out as
 * bm_tc_conv1d.  stats (nullable; plain forward only): BatchNorm batch statistics stats[0:Ntot] = sum(y), stats[Ntot:2Ntot]
 * = sum(y^2) (fp64, zeroed by the call) accumulated in shared memory across the CTA's tiles -- replaces bm_col_stats.
 * Shape gate (bm_tc_conv1d_persistent_supported): Cin % 32 == 0 and Ntot % 320 == 0 or Ntot % 256 == 0 (GLU: halves). */
int bm_tc_conv1d_persistent_supported(int T, int Cin, int Ntot, int Kw, int glu);
int bm_tc_conv1d_persistent(const float* x, const float* w_raw, const float* bias, int accumulate, int B, int T, int Cin,
                            int Ntot, int Kw, int dilation, int sign, int glu, int act, int out_tmajor, float* y,
                            float* aux, float* glu_out, double* stats, int* status, bm_stream_t stream);

/* The same conv on the F16 tensor pipe (csrc/tc_convh.cuh; replaces the same reference lines as bm_tc_conv1d_persistent:
 * nn.Conv1d / GLU in bm/models/common.py:107-151, the head's 1x1 convs simpleconv.py:153-168).  Each fp32 operand is
 * carried as two fp16 pieces (11 + 11 significant bits, like the two tf32 pieces) of the tensor times a power of two that
 * puts its largest magnitude in [2^14, 2^15): three kind::f16 MMAs per product cost half the tensor-pipe time of three
 * kind::tf32 MMAs.  bm_amax: amax[0] = max |x[i]| (device float; one HBM pass).  bm_f16_split: hi/lo = fp16 pieces of
 * src * scale(amax[0]) in the same element order (the weights, once per step, from bm_tc_weight_split's raw K-major
 * re-layout).  bm_tc_conv1d_f16: arguments as bm_tc_conv1d_persistent with (w_hi, w_lo, w_amax) in place of w_raw and
 * x_amax = the device float bm_amax wrote for x; same shape gate. */
int bm_amax(const float* x, long long n, float* amax, bm_stream_t stream);
int bm_f16_split(const float* src, long long n, const float* amax, void* hi, void* lo, bm_stream_t stream);
/* bm_tc_weight_split_f16: bm_tc_weight_split + bm_f16_split in one launch: w [Cout,Cin,Kw] (nn.Conv1d layout) times
 * scale(w_amax[0]) -> fp16 pieces of the forward operand f [Kw,Cout,Cin] and of the data-gradient operand g [Kw,Cin,Cout]
 * (either pair may be NULL); w_amax = bm_amax over w. */
int bm_tc_weight_split_f16(const float* w, const float* w_amax, int Cout, int Cin, int Kw, void* f_hi, void* f_lo, void* g_hi,
                           void* g_lo, bm_stream_t stream);
int bm_tc_conv1d_f16(const float* x, const float* x_amax, const void* w_hi, const void* w_lo, const float* w_amax,
                     const float* bias, int accumulate, int B, int T, int Cin, int Ntot, int Kw, int dilation, int sign,
                     int glu, int act, int out_tmajor, float* y, float* aux, float* glu_out, double* stats,
                     float* amax_out /* nullable: max |glu_out| (glu) or max |y| (act), see bm_bn_gelu_skip_fwd */, int* status,
                     bm_stream_t stream);

/* bm_tc_wgrad: weight gradient on the tensor cores (3xTF32): dw[m][n][tap] = sum_{b,t} dy[b,t,m] x[b,t+(tap-Kw/2)*dil,n]
 * for n < Ntrue (x may be channel-padded to N); dy [B,T,M], x [B,T,N] channels-last; dw in nn.Conv1d layout
 * [M][Ntrue][Kw].  workspace: bm_tc_wgrad_workspace() floats (per-batch-slice partial tiles, reduced in a fixed
 * order => deterministic).  dbias (nullable) [M] receives the bias gradient sum_{b,t} dy[b,t,m], accumulated from the dy
 * values the kernel already holds in registers.  bm_col_sum: out[c] = sum_r x[r,c] (other bias gradients). */
int bm_tc_wgrad_supported(int M, int N);
long long bm_tc_wgrad_workspace(int B, int M, int N, int Kw);
int bm_tc_wgrad(const float* dy, const float* x, int B, int T, int M, int N, int Ntrue, int Kw, int dilation,
                float* workspace, float* dw, float* dbias, int* status, bm_stream_t stream);
/* bm_tc_wgrad_conv: the same weight gradient on CTA PAIRS (csrc/tc_wgradp.cuh): ONE GEMM whose output rows are the
 * (tap, x-channel) pairs (3 x 320 = 960 rows in 4 pair-tiles instead of 3 x 384 padded rows), reduced over the flattened
 * rows b*T + t in exact chunks of 32 (the tap shift is applied to the x side; a shifted row across a sample edge reads 0),
 * each CTA holding half of the dy tile.  No dbias output.  T >= 32; M % 64 == 0; N % 4 == 0. */
int bm_tc_wgrad_conv_supported(int T, int M, int N, int Kw);
long long bm_tc_wgrad_conv_workspace(int B, int T, int M, int N, int Kw);
int bm_tc_wgrad_conv(const float* dy, const float* x, int B, int T, int M, int N, int Ntrue, int Kw, int dilation,
                     float* workspace, float* dw, int* status, bm_stream_t stream);
/* bm_tc_wgrad_conv_f16: the same on the F16 pipe (csrc/tc_wgradh.cuh; see bm_tc_conv1d_f16 for the arithmetic): both
 * operands as fp16 hi/lo pieces of the tensors scaled by powers of two from dy_amax / x_amax (device floats: bm_amax or a
 * producer's amax_out); the dY tile is transposed to K-major rows while it is split.  Same gate and workspace. */
int bm_tc_wgrad_conv_f16(const float* dy, const float* dy_amax, const float* x, const float* x_amax, int B, int T, int M,
                         int N, int Ntrue, int Kw, int dilation, float* workspace, float* dw, int* status,
                         bm_stream_t stream);
int bm_col_sum(const float* x, long long rows, int C, float* out, bm_stream_t stream);
/* SubjectLayers (common.py:55-58) on the tensor cores.
 * bm_tc_pointwise_sel: y[b,t,n] = sum_k x[b,t,k] W[wsel[b]][n][k] with tf32-split weight sets w_hi/w_lo [S][Ntot][Cin].
 * bm_tc_wgrad_grouped: out[g][m][n] = sum_{b in group g} sum_t dy[b,t,m] x[b,t,n], groups as CSR (order, seg_off[G+1]);
 * out is [G][ceil(M/128)*128][N] (rows >= M are zero). */
int bm_tc_pointwise_sel(const float* x, const float* w_hi, const float* w_lo, const int* wsel, int n_sets, int B, int T,
                        int Cin, int Ntot, float* y, int* status, bm_stream_t stream);
int bm_tc_wgrad_grouped(const float* dy, const float* x, const int* order, const int* seg_off, int G, int B, int T, int M,
                        int N, float* out, int* status, bm_stream_t stream);
/* dh = dq * GELU'(h), elementwise over n values (dh may alias dq): the head's activation backward. */
int bm_gelu_bwd(const float* dq, const float* h, long long n, float* dh, bm_stream_t stream);
/* y[b,c,t] = x[b,c,t] * mask[c]: SimpleConv(subsample_meg_channels=n) keeps n sensors drawn with random.Random(1234)
 * and zeroes the others before the merger (bm/models/simpleconv.py:97-102, 200-203).  y may alias x. */
int bm_channel_mask(const float* x, const float* mask, int B, int C, int T, float* y, bm_stream_t stream);
/* in [Z,N,T] (channel-major) -> out [Z,T,N] (channels-last): the gradient of `estimate` enters the head backward. */
int bm_transpose_nt(const float* in, int Z, int N, int T, float* out, bm_stream_t stream);
/* same with an output row stride ld_out >= N (pad columns written as zeros): meg [B,C,T] -> channels-last, channel-padded. */
int bm_transpose_nt_ld(const float* in, int Z, int N, int T, int ld_out, float* out, bm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BM_B200_H_ */
