/* caphn_b200.h -- C-ABI of libcaphn_b200.so: the B200 (sm_100a) hot path of Caption-HN.
 *
 * The reference (zacharie12/Hypernet-image-captioning) is pure Python: it has no FFI/plugin boundary of its own, its
 * "kernels" are torch.nn calls.  This header is therefore the boundary a reference maintainer would bind (ctypes
 * stub in INTEGRATION.md); every entry point names the reference lines whose torch calls it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers (fp32 unless noted; token ids are int64 = torch.long), caller-allocated;
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it (no sync, no allocation);
 *   - return value: 0 = ok, -1 = invalid argument, otherwise the cudaError_t of the failed launch;
 *   - "time-major" sequence tensors have row index t*B + b; "batch-major" b*T + t;
 *   - `long` is 64-bit (LP64).
 */
#ifndef CAPHN_B200_H
#define CAPHN_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- hypernetwork layers (hypernet_attention.py:111-118, hypernet.py:104-111; nn.Linear + nn.LeakyReLU) ----------- */

/* Y[g*ldy+n] = act(sum_k A[g*lda+k] * W[n*K+k] + bias[n]), g < G <= 8.  act: 0 none, 1 LeakyReLU(slope).
 * W is streamed exactly once (HBM-bound); Y may be a column slice of theta (ldy = theta length).  W 16-byte aligned. */
int caphn_rows_linear_fwd(const float* W, const float* bias, const float* A, long lda, float* Y, long ldy, int G,
                          long N, long K, int act, float slope, void* stream);

/* Backward of the above (autograd of the same reference lines).  dP: scratch [G,N].  dW[N,K], dbias[N] are written;
 * dA[g*ldda+k] is accumulated with atomics (caller zero-initialises; NULL skips it).  Y only read when act == 1.
 * One pass: reads W once, writes dW once.  G <= 64. */
int caphn_rows_linear_bwd(const float* W, const float* A, long lda, const float* Y, long ldy, const float* dY,
                          long lddy, float* dP, float* dW, float* dbias, float* dA, long ldda, int G, long N, long K,
                          int act, float slope, void* stream);

/* bf16-weight variants (bf16 mode): W, dW are bf16 [N,K]; bias, A, Y, dY, dP, dbias, dA stay fp32; fp32 accumulation;
 * dW rounded to bf16 on store.  Half the HBM bytes. */
int caphn_rows_linear_fwd_bf16(const void* W, const float* bias, const float* A, long lda, float* Y, long ldy, int G,
                               long N, long K, int act, float slope, void* stream);
int caphn_rows_linear_bwd_bf16(const void* W, const float* A, long lda, const float* Y, long ldy, const float* dY,
                               long lddy, float* dP, void* dW, float* dbias, float* dA, long ldda, int G, long N,
                               long K, int act, float slope, void* stream);

/* ---- dense fp32 GEMM (addmm behind nn.Linear / nn.GRUCell: models/decoderlstm.py:61,100,105; later.py:411,418,442) -- */

/* C[m*ldc+n] = sum_k A(m,k) B(n,k) (+bias[n]) (ReLU).  A(m,k) = a_kmajor ? A[m*lda+k] : A[k*lda+m]; same for B.
 * splitk > 1 or accumulate != 0: result is atomically added into C. */
int caphn_gemm_f32(const float* A, long lda, int a_kmajor, const float* B, long ldb, int b_kmajor, float* C, long ldc,
                   const float* bias, int M, int N, int K, int relu, int splitk, int accumulate, void* stream);

/* ---- tensor-core GEMM (tcgen05 + TMEM + TMA), same reference call sites as caphn_gemm_f32 for the large products --- */

/* Split fp32 into the bf16x3 operand format: hi = rn(x), lo = rn(x - hi), both [R, Kp] bf16 row-major, Kp % 64 == 0,
 * columns [C, Kp) zero.  lo == NULL: hi only (plain bf16 mode).  The _t variant transposes: src [R,C] -> hi/lo [C, Rp]. */
int caphn_split_bf16(const float* src, long lds, long R, int C, void* hi, void* lo, long Kp, void* stream);
int caphn_split_bf16_t(const float* src, long lds, int R, int C, void* hi, void* lo, long Rp, void* stream);
/* C[M,N] (fp32, ldc) = A B^T (+bias[n]) (ReLU); A = (Ahi, Alo) [M,Kp], B = (Bhi, Blo) [N,Kp] in the split format.
 * Three MMAs per k-slice (hi*hi + hi*lo + lo*hi) with fp32 accumulation in TMEM: ~1e-5 relative, fp32-class.
 * Alo == Blo == NULL: single bf16 MMA per k-slice.  splitk: 0 = automatic, 1 = none, > 1 = split the K loop over more
 * CTAs and add the partial tiles atomically (C is zeroed by the call; not combinable with ReLU). */
int caphn_gemm_tc(const void* Ahi, const void* Alo, const void* Bhi, const void* Blo, long Kp, float* C, long ldc,
                  const float* bias, int M, int N, int relu, int splitk, void* stream);

/* General operand layouts: x_mn = 0: K-major hi/lo [rows, K] with row pitch x_ld; x_mn = 1: MN-major hi/lo [K rows, MN cols]
 * with row pitch x_ld, i.e. the operand of a transposed product (dW = dY^T X) is read in place (UMMA MN-major shared-memory
 * descriptors + 64x64 TMA boxes), no transposed copy.  x_ld % 8 == 0. */
int caphn_gemm_tc_ex(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                     int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, int relu, int splitk,
                     void* stream);

/* dst[c*ldd+r] = src[r*lds+c] (zero padded to ldd) / dst[r*ldd+c] = src[r*lds+c] (zero padded): lay generated
 * weights out with 16-byte rows for the recurrence kernels. */
int caphn_transpose_pad(const float* src, long lds, float* dst, long ldd, int R, int C, void* stream);
int caphn_copy_pad(const float* src, long lds, float* dst, long ldd, long R, int C, void* stream);
/* The same for nb matrices in one launch: matrix z is read at src + z*sstride and written at dst + z*dstride (floats) --
 * e.g. the per-group W_hh packs of a many-style batch, read straight out of Theta [G, theta] (sstride = theta). */
int caphn_transpose_pad_batched(const float* src, long sstride, long lds, float* dst, long dstride, long ldd, int nb,
                                int R, int C, void* stream);
int caphn_copy_pad_batched(const float* src, long sstride, long lds, float* dst, long dstride, long ldd, int nb, long R,
                           int C, void* stream);

/* ---- pooled-feature decoder recurrence (later.py:389-490 DecoderGRU; torch GRUCell gates r,z,n) -------------------- */

/* All T steps (and all layers) in one launch.  GI [T,B,3H] = x_t W_ih^T + b_ih of layer 0 (time-major); WhhT [H,ld3]
 * (= W_hh^T, ld3 % 4 == 0); Hall [T+1,B,H] with Hall[0] = h0 on entry, Hall[t+1] = h_t (last layer) on exit; Hbm [B,T,H]
 * optional batch-major copy.  Extra layers (num_layers > 1, later.py:413-414 `h = layer(h, h)`): `extra` is a HOST array
 * of 4*(NL-1) device pointers {WihT_l, WhhT_l, bih_l, bhh_l}.  saved [NL][4][T,B,H] (R,Z,N,GHN) and Hmid [NL-1][T,B,H]
 * (outputs of the lower layers) are written for the backward when non-NULL. */
int caphn_gru_seq_fwd(const float* GI, const float* WhhT, int ld3, const float* bhh, float* Hall, float* Hbm,
                      float* saved, float* Hmid, const void* const* extra, int NL, int B, int T, int H, void* stream);

/* BPTT.  dHbm [B,T,H] = dL/dh_t from the vocabulary projection; Whh [3H,ldh]; `extra` = HOST array of 2*(NL-1) device
 * pointers {Wih_l, Whh_l} ([3H,ldh]).  Outputs dGI,dGH [T,B,3H] (layer 0), xdGI,xdGH [NL-1][T,B,3H], dh0 [B,H]. */
int caphn_gru_seq_bwd(const float* dHbm, const float* saved, const float* Hall, const float* Hmid, const float* Whh,
                      int ldh, const void* const* extra, float* dGI, float* dGH, float* xdGI, float* xdGH, float* dh0,
                      int NL, int B, int T, int H, void* stream);

/* Weights-resident variant (single layer): W_hh [3H,H] (plain row-major) is loaded ONCE into shared memory, split by hidden
 * unit over a thread-block cluster; h is exchanged through DSMEM every step.  caphn_gru_cluster_plan: *cs = cluster size
 * used for hidden size H (0: does not fit -> use caphn_gru_seq_*).  saved = [4][T,B,H] or NULL. */
int caphn_gru_cluster_plan(int H, int* cs);
int caphn_gru_cluster_fwd(const float* GI, const float* Whh, const float* bhh, float* Hall, float* Hbm, float* saved,
                          int B, int T, int H, void* stream);
int caphn_gru_cluster_bwd(const float* dHbm, const float* saved, const float* Hall, const float* Whh, float* dGI,
                          float* dGH, float* dh0, int B, int T, int H, void* stream);

/* ---- attention decoder recurrence (models/decoderlstm.py:78-108 AttentionGru loop; models/attention.py:21-46) ------- */

/* Steps [t0,t1) of: u = U_a h + b_u; s_p = v_a.tanh(K_p + u) + b_v; alpha = softmax_p s; ctx = sum_p alpha_p f_p;
 * h' = GRUCell([x_w, ctx], h) with the word half of the input projection precomputed (GIw [T,B,3H], incl. b_ih).
 * Kp [B,P,H] = W_a f + b_a (hoisted, attention.py:34); f [B,P,F]; UaT [H,ldh] = U_a^T; WihcT [F,ld3] = W_ih[:,E:]^T;
 * WhhT [H,ld3] = W_hh^T.  Hall [T+1,B,H] (Hall[t0] = previous state on entry); Hbm [B,T,H] optional; attn [B,T,P];
 * ctx rows at ctx + (t*B+b)*ldctx; Upre,R,Z,Nn,GHN [T,B,H] saved for the backward (all or none). */
int caphn_attgru_seq_fwd(const float* Kp, const float* f, const float* GIw, const float* UaT, const float* bu,
                         const float* va, const float* bv, const float* WihcT, const float* WhhT, const float* bhh,
                         float* Hall, float* Hbm, float* attn, float* ctx, long ldctx, float* Upre, float* R, float* Z,
                         float* Nn, float* GHN, int B, int T, int P, int H, int F, int ldh, int ld3, int t0, int t1,
                         void* stream);
/* BPTT of the above over all T steps (SURVEY Appendix B.2-B.4).  Ua [H,ldh], Wihc [3H,ldf] = W_ih[:,E:], Whh [3H,ldh].
 * Outputs dGI,dGH [T,B,3H], dU [T,B,H], dCTX [T,B,F], dh0 [B,H]; dK [B,P,H], dva [H], dbv [1] are accumulated
 * (zero-initialised by the caller).  dattn [B,T,P] (gradient of the returned attention weights) may be NULL. */
int caphn_attgru_seq_bwd(const float* dHbm, const float* dattn, const float* Kp, const float* f, const float* attn,
                         const float* Upre, const float* R, const float* Z, const float* Nn, const float* GHN,
                         const float* Hall, const float* Ua, const float* va, const float* Wihc, const float* Whh,
                         float* dGI, float* dGH, float* dU, float* dCTX, float* dK, float* dva, float* dbv, float* dh0,
                         int B, int T, int P, int H, int F, int ldh, int ldf, void* stream);
/* LSTM recurrence of the pooled variant's DecoderRNN (hypernet.py:53 with type != 'gru'; later.py:254-324 forward,
 * :326-360 infer): torch nn.LSTMCell, gate order i,f,g,o, zero initial (h, c); extra layers as (h,c) = layer(h,(h,c))
 * (later.py:279-281).  GI [T,B,4H] = layer-0 input projection incl. b_ih; WhhT [H,ld4] k-major; Hall [T+1,B,H] with
 * Hall[0] = h0; c0 / cT [B,H] = cell state in / out (NULL: zeros / not returned); `extra` = HOST array of 4*(NL-1)
 * device pointers {WihT_l, WhhT_l, bih_l, bhh_l}; saved [NL][6][T,B,H].
 * Backward: Whh [4H,ldh] row-major padded, `extra` = HOST array of 2*(NL-1) pointers {Wih_l, Whh_l}; dG [NL][T,B,4H]. */
int caphn_lstm_seq_fwd(const float* GI, const float* WhhT, int ld4, const float* bhh, float* Hall, float* Hbm,
                       float* saved, float* Hmid, const void* const* extra, const float* c0, float* cT, int NL, int B,
                       int T, int H, void* stream);
int caphn_lstm_seq_bwd(const float* dHbm, const float* saved, const float* Whh, int ldh, const void* const* extra,
                       float* dG, float* dh0, int NL, int B, int T, int H, void* stream);
/* Single-layer LSTM recurrence of a many-style batch (pooled DecoderRNN with per-row style groups): rows sorted by group,
 * CTA i runs tiles[i] = {first row, rows 1..4, group, 0} (int32, 16-byte aligned; a tile never straddles two groups) with
 * that group's weights: forward WhhT pack [G][H][ld4] and b_hh at bhh + group*bstride, backward Whh pack [G][4H][ldh].
 * h0 = Hall[0], c0 = zeros; saved [6][T,B,H], dG [T,B,4H], cT / dh0 [B,H] as in the single-style calls.  Each row
 * computes exactly what caphn_lstm_seq_fwd / _bwd compute for it. */
int caphn_lstm_seq_fwd_grouped(const float* GI, const float* WhhT, int ld4, const float* bhh, long bstride, float* Hall,
                               float* Hbm, float* saved, float* cT, int B, int T, int H, const int* tiles, int ntiles,
                               void* stream);
int caphn_lstm_seq_bwd_grouped(const float* dHbm, const float* saved, const float* Whh, int ldh, float* dG, float* dh0,
                               int B, int T, int H, const int* tiles, int ntiles, void* stream);
/* Step-split forward (default for H, F <= 208): three batch-wide launches per time step instead of one persistent
 * kernel, chained with programmatic dependent launch -- U: u = U_a h + b_u on the warp tensor cores (bf16 hi/lo split,
 * fp32 accumulate); A: one CTA per batch row, K_b / f_b fetched into shared memory by bulk TMA copies, scores, softmax,
 * ctx; Y: gi_ctx / gh on the warp tensor cores + the r/z/n gates.  Replaces the same reference lines as
 * caphn_attgru_seq_fwd (models/decoderlstm.py:97-100, models/attention.py:33-45).
 * caphn_attstep_pack_size: *pack_bytes = size of the weight pack (0: shape not covered, use caphn_attgru_seq_fwd),
 *   *work_bytes = size of the scratch buffer for batch B (u and the bf16 hi/lo operand rows passed between the kernels).
 * caphn_attstep_pack: builds the mma-fragment-ordered bf16 hi/lo pack of Wih[:, E:E+F], Whh (plain row-major
 *   [3H,E+F], [3H,H]) and Ua [H,H]; once per generated theta.
 * caphn_attstep_fwd: steps [t0,t1); tensors as in caphn_attgru_seq_fwd.  work: 256-byte aligned.  resume != 0: the
 *   previous call ran up to step t0 on the same work / Hall buffers (one-step-per-call decode), skip the re-conversion
 *   of Hall[t0]. */
int caphn_attstep_pack_size(int H, int F, int P, int B, long* pack_bytes, long* work_bytes);
int caphn_attstep_pack(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, void* pack,
                       void* stream);
int caphn_attstep_fwd(const float* Kp, const float* f, const float* GIw, const float* bu, const float* va,
                      const float* bv, const void* pack, void* work, const float* bhh, float* Hall, float* Hbm,
                      float* attn, float* ctx, long ldctx, float* Upre, float* R, float* Z, float* Nn, float* GHN, int B,
                      int T, int P, int H, int F, int t0, int t1, int resume, void* stream);
/* Step-split BPTT (default when covered): the backward of caphn_attstep_fwd as three launches per time step --
 * G1: dh_t (du_{t+1} U_a on the warp tensor cores + carries) and the GRU gate gradients; G2: dctx_t = dgi_t W_ih[:,E:]
 * and dgh_t W_hh on the warp tensor cores; A': attention backward per row (K_b / f_b tiles by bulk TMA) -- plus one
 * deferred kernel for dK and dv_a.  Same tensors and results as caphn_attgru_seq_bwd; dK / dva / dbv need no
 * zero-initialisation.
 * caphn_attstep_bwd_size: *pack_bytes (0: shape not covered, use caphn_attgru_seq_bwd), *work_bytes for (B, T).
 * caphn_attstep_bwd_pack: transposed-weight fragment pack of U_a, Wih[:, E:E+F], Whh (plain row-major). */
int caphn_attstep_bwd_size(int H, int F, int P, int B, int T, long* pack_bytes, long* work_bytes);
int caphn_attstep_bwd_pack(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, void* pack,
                           void* stream);
int caphn_attstep_bwd(const float* dHbm, const float* dattn, const float* Kp, const float* f, const float* attn,
                      const float* Upre, const float* R, const float* Z, const float* Nn, const float* GHN,
                      const float* Hall, const float* va, const void* pack, void* work, float* dGI, float* dGH,
                      float* dU, float* dCTX, float* dK, float* dva, float* dbv, float* dh0, int B, int T, int P, int H,
                      int F, void* stream);
/* df[b,p,:] += sum_t attn[b,t,p] * dCTX[t,b,:]  (context-vector backward, deferred out of the BPTT loop). */
int caphn_attn_df(const float* attn, const float* dCTX, float* df, int B, int T, int P, int F, void* stream);

/* ---- loss / sampling / embedding (cc_train_hypernet.py:153, hypernet.py:145; decoderlstm.py:62,91-96; later.py:472-479) */

/* Mean softmax cross-entropy over rows of X[M,V] whose target != ignore (when has_ignore).  lse [M]; scratch [2M];
 * lossbuf[0] = mean loss, lossbuf[1] = number of counted rows. */
int caphn_ce_fwd(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                 float* lse, float* scratch, float* lossbuf, void* stream);
/* dX = gscale[0] * d(mean loss)/dX, using lse / lossbuf from caphn_ce_fwd (no host sync). */
int caphn_ce_bwd(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                 const float* lse, const float* gscale, const float* lossbuf, float* dX, long lddx, void* stream);
/* Same gradient, written directly as tensor-core operands (no fp32 dlogits): hi/lo [M,Vp] = split(d), hiT/loT [V,Mp] =
 * split(d^T) (Vp, Mp multiples of 64), dbias[v] += sum_m d[m,v] (zero-initialised by the caller). */
int caphn_ce_bwd_split(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                       const float* lse, const float* gscale, const float* lossbuf, void* hi, void* lo, long Vp,
                       void* hiT, void* loT, long Mp, float* dbias, void* stream);
/* Y (optional) = row softmax of X[M,V]; amax (optional, int64) = row argmax, lowest index on ties, NaN counted as -inf
 * (an all-NaN / all -inf row gives 0). */
int caphn_softmax_argmax(const float* X, long ld, long M, int V, float* Y, long ldy, long long* amax, void* stream);
/* out[i,:] = table[idx[i],:]  (idx int64; negative idx -> zero row). */
int caphn_gather_rows(const float* table, const long long* idx, long n, int E, float* out, long ldo, void* stream);
/* Time-major decoder inputs X[T,B,E].  mode 0 (later.py:411,418): X[0]=feat, X[t]=Emb[caps[:,t-1]];
 * mode 1 (models/decoderlstm.py:82-88): X[0]=X[1]=0, X[t]=Emb[caps[:,t-1]]. */
int caphn_build_inputs(const float* feat, const float* emb, const long long* caps, int B, int T, int E, int mode,
                       float* X, void* stream);
/* dEmb[caps[b,t-1],:] += dX[t,b,:] for t >= t0  (embedding_dense_backward). */
int caphn_embed_scatter_add(const float* dX, const long long* caps, int B, int T, int E, int t0, float* dEmb,
                            void* stream);
/* table[idx[i],:] += dX[i*ldx + :]  for idx[i] >= 0  (embedding backward for arbitrary fed-back tokens). */
int caphn_scatter_add_rows(const float* dX, long ldx, const long long* idx, long n, int E, float* table, void* stream);
/* out[n] += sum_m X[m*ld+n]  (bias gradients). */
int caphn_colsum(const float* X, long ld, long M, int N, float* out, void* stream);
/* out[b,f] = mean_p X[b,p,f] (models/decoderlstm.py:133) and its backward dX[b,p,f] += g[b,f]/P (+ extra[b,p,f] when
 * extra != NULL: a second gradient contribution to the same tensor folded into the same pass). */
int caphn_mean_pos(const float* X, int B, int P, int Fd, float* out, void* stream);
int caphn_mean_pos_bwd(const float* g, const float* extra, int B, int P, int Fd, float* dX, void* stream);
/* y[i] = ref[i] > 0 ? y[i] : 0  (ReLU backward, in place). */
int caphn_relu_mask(const float* ref, float* y, long n, void* stream);

/* ---- bookkeeping -------------------------------------------------------------------------------------------------- */
/* ---- optimizer step (SURVEY.md section 8(f) rank 1) -------------------------------------------------------------------
 * torch.optim.Adam(params, lr) of cc_train_hypernet.py:110-122 / hypernet.py:116-123 and Lightning's
 * gradient_clip_val=5. (cc_train_hypernet.py:405 = torch.nn.utils.clip_grad_norm_), as single-pass HBM streaming kernels.
 * caphn_sumsq: *sumsq (device double) += sum x[i]^2.   caphn_clip_coef: *coef = min(1, max_norm / (sqrt(*sumsq) + 1e-6)).
 * caphn_adam_step: one Adam step on a flat fp32 tensor (amsgrad=False); step is 1-based; gscale (device scalar or NULL)
 * multiplies the gradient on the fly (the clip coefficient -- the stored gradient is not modified). */
int caphn_sumsq(const float* x, long n, double* sumsq, void* stream);
int caphn_clip_coef(const double* sumsq, float max_norm, float* coef, float* norm, void* stream);
int caphn_adam_step(float* p, const float* g, float* m, float* v, long n, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int step, const float* gscale, void* stream);
/* Rank-G form of the head-weight gradient (dW = dP^T A, G = #style groups <= 4; caphn_rows_linear_bwd with dW == NULL
 * leaves it in that form): its squared norm from two G x G Gram matrices, and the Adam step that forms g[n,k] on the fly
 * -- 24 bytes per parameter instead of 8 (dW write + norm read) + 28.
 * caphn_gram: out[G*G] (device double, caller-zeroed) += X X^T, X [G,L] row stride ld.
 * caphn_sumsq_lowrank: *sumsq += sum_{q,r} gram_dp[q,r] * gram_a[q,r] = ||dP^T A||_F^2. */
int caphn_gram(const float* X, long ld, int G, long L, double* out, void* stream);
int caphn_sumsq_lowrank(const double* gram_dp, const double* gram_a, int G, double* sumsq, void* stream);
int caphn_adam_step_lowrank(float* p, float* m, float* v, const float* dP, long ldp, const float* A, long lda, int G,
                            long N, long K, double lr, double beta1, double beta2, double eps, double weight_decay,
                            int step, const float* gscale, void* stream);

/* ---- caption metrics, token-level part (csrc/metrics.cu) ------------------------------------------------------------
 * Replaces the per-token `.item()` loops of utils.py:161-190 (cap_to_text / cap_to_text_gt) that metric_score
 * (utils.py:229-262) runs inside every training_step (cc_train_hypernet.py:154).
 * out[b, :len[b]] = tokens of tok[b, :T] (row stride ldt) that are neither pad nor start, up to (excluding) the first end
 * token; out[b, len[b]:] = pad.  out is [B,T] int64, len is [B] int32. */
int caphn_caption_compact(const long long* tok, long ldt, int B, int T, long long pad, long long start, long long end,
                          long long* out, int* len, void* stream);
/* Corpus-BLEU sufficient statistics (the `datasets` "bleu" metric == tensorflow/nmt compute_bleu, requested with
 * max_order 1..4 at utils.py:250-258) of B (hypothesis, single reference) pairs of compacted captions hyp [B,Th] /
 * ref [B,Tr] int64 with lengths int32, ADDED into counts[2*max_order + 2] (uint64, zeroed by the caller): clipped n-gram
 * matches per order, candidate n-grams per order, total hypothesis length, total reference length.  max_order <= 4. */
int caphn_bleu_counts(const long long* hyp, const int* hyp_len, int Th, const long long* ref, const int* ref_len, int Tr,
                      int B, int max_order, unsigned long long* counts, void* stream);

/* *out = number of CUDA kernels launched by this library so far (host-side counter). */
int caphn_launch_count(unsigned long long* out);
/* *out = 100 (library compiled for sm_100a). */
int caphn_build_arch(int* out);

/* ------------------------------------------------------------------------------------------------------------------
 * Many-style ("grouped") path: one batch whose rows use G different generated weight sets -- BASELINE.json configs[3]
 * (Conceptual-Captions domains) and the north star's "per-style grouped GEMM".  Reference semantics: one
 * HyperNet.forward + captioner call per sample's style (train_cc.py:90-123); cc_train_hypernet.py:134-153 is the G = 1
 * special case.  The batch is sorted by group; the recurrence keeps the time-major layout, the time-batched products
 * run as ONE grouped tensor-core launch each.
 *
 * caphn_gemm_tc_grouped: num_units output tiles, unit i described by 12 int32 words
 *   {a_row, b_row, ka0, kb0, nkb, m_valid, n_valid, bias_off, map0, c_off_lo, c_off_hi, 0}: the tile multiplies A rows
 *   a_row.. (128) with B rows b_row.. (BN) over nkb 64-wide k blocks starting at ka0 in A and kb0 in B, and writes
 *   C + c_off (+ bias[bias_off + col]) or, with rowmap, tile row r to C row rowmap[map0 + r] (negative: skip).
 *   Operands: 2-D bf16 arrays (hi, optional lo), x_inner contiguous elements per row, x_outer rows, pitch x_ld; K-major
 *   (x_mn = 0: inner = K) or MN-major (x_mn = 1: inner = operand rows, outer = K).  Replaces, for all groups at once, the
 *   addmm of nn.GRUCell's input projection (models/decoderlstm.py:100) and its three backward products.
 * caphn_split_bf16_gather / _batched: build those operands (bf16 hi/lo) while permuting rows between the time-major and
 *   the group-major order / collecting the W_ih block of every row of Theta [G, theta].
 * caphn_group_colsum: per-group bias gradients.
 * caphn_attstep_pack_grouped / caphn_attstep_fwd_grouped / caphn_attstep_bwd_pack_grouped / caphn_attstep_bwd_grouped:
 *   the step-split recurrence with one weight pack per group; `tiles` = {first row, rows, group, 0} records (int32 x 4,
 *   16-byte aligned) that never straddle a group (<= 64 rows forward, <= 32 backward); tile_rows = the largest row count in
 *   the table (<= 8 selects small-tile kernels: many CTAs per SM hide the per-group weight loads of a many-domain batch).
 * ------------------------------------------------------------------------------------------------------------------ */
int caphn_gemm_tc_grouped(const void* Ahi, const void* Alo, long a_inner, long a_outer, long a_ld, int a_mn,
                          const void* Bhi, const void* Blo, long b_inner, long b_outer, long b_ld, int b_mn, float* C,
                          long ldc, const float* bias, const int* rowmap, const void* units, int num_units, int BN,
                          void* stream);
int caphn_split_bf16_gather(const float* src, long lds, const int* rowmap, long R, int C, void* hi, void* lo, long Kp,
                            void* stream);
int caphn_split_bf16_batched(const float* src, long sstride, long lds, int nb, int R, int C, void* hi, void* lo, long Kp,
                             void* stream);
int caphn_group_colsum(const float* X, long ldx, const int* goff, int G, int B, int T, int N, float* out, long ldo,
                       void* stream);
/* nn.LeakyReLU(slope) forward (in place on y) / backward (in place on dy, y = activation output) for the many-group
 * hypernet, whose layers run as dense tensor-core GEMMs instead of the weight-streaming kernels. */
int caphn_leaky_relu(float* y, long n, float slope, void* stream);
int caphn_leaky_relu_bwd(const float* y, float* dy, long n, float slope, void* stream);
int caphn_attstep_pack_grouped(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, int G,
                               long gstride, void* pack, void* stream);
int caphn_attstep_fwd_grouped(const float* Kp, const float* f, const float* GIw, const float* bu, const float* va,
                              const float* bv, const void* pack, void* work, const float* bhh, float* Hall, float* Hbm,
                              float* attn, float* ctx, long ldctx, float* Upre, float* R, float* Z, float* Nn, float* GHN,
                              int B, int T, int P, int H, int F, int t0, int t1, int resume, const int* tiles, int ntiles,
                              int tile_rows, void* stream);
int caphn_attstep_bwd_pack_grouped(const float* Wih, const float* Whh, const float* Ua, int E, int F, int H, int G,
                                   long gstride, void* pack, void* stream);
int caphn_attstep_bwd_grouped(const float* dHbm, const float* dattn, const float* Kp, const float* f, const float* attn,
                              const float* Upre, const float* R, const float* Z, const float* Nn, const float* GHN,
                              const float* Hall, const float* va, const void* pack, void* work, float* dGI, float* dGH,
                              float* dU, float* dCTX, float* dK, float* dva, float* dbv, float* dh0, int B, int T, int P,
                              int H, int F, const int* tiles, int ntiles, int tile_rows, void* stream);

/* Batched device-resident beam search bookkeeping (HyperNet.test_step, hypernet_attention.py:247-326): for B images x k
 * beams (rows b*k.., live beams first) one launch does what the reference does on the host between two decoder steps --
 * log-softmax + running scores, top-k_live over (live rows x V) (step 1: row 0 only), completed beams moved to the image's
 * complete list, survivors compacted with their history / score / hidden state, next input words (-1 = zero embedding).
 * step is 1-based; last != 0: images with beams still open are flagged in failed[] (the reference returns no caption).
 * k <= V (else CAPHN_EINVAL).  A row whose log-sum-exp is not finite (a NaN / +inf logit) offers no candidates; an image
 * left with fewer eligible candidates than live beams ends at once with failed[b] = 1, live[b] = 0. */
int caphn_beam_step(const float* logits, const float* h_out, float* h_next, float* scores, int* live, int* prev_tok,
                    long long* words, const int* seq_in, int* seq_out, float* comp_score, int* comp_seq, int* comp_len,
                    int* ncomp, int* failed, int B, int k, int V, int H, int L, int step, int end_tok, int last,
                    void* stream);

/* bf16 mode of the optimizer (hypernet.set_precision("bf16")): the parameter and its gradient are bf16 (what the
 * weight-streaming kernels read and write), the master weight and the Adam moments stay fp32.  caphn_sumsq_bf16 is the
 * norm pass over a bf16 gradient; caphn_adam_step_bf16 is caphn_adam_step on (master, m, v) with p = bf16(master). */
int caphn_sumsq_bf16(const void* x, long n, double* sumsq, void* stream);
int caphn_adam_step_bf16(void* p, const void* g, float* master, float* m, float* v, long n, double lr, double beta1,
                         double beta2, double eps, double weight_decay, int step, const float* gscale, void* stream);

/* Greedy decode (models/decoderlstm.py:89-96: top_idx = topk(log_softmax(output / 0.5), 1) == arg-max of the logits):
 * caphn_gemm_tc_amax = caphn_gemm_tc_ex whose epilogue also reduces every row of every output tile to (max, column)
 * partials [M, amax_ld] (*nparts slots are written; amax_ld >= 2*ceil(N/128) suffices); caphn_argmax_finish_gather
 * finishes the arg-max (lowest column on ties; NaN never wins; 0 for a row with no candidate), writes the token and gathers
 * the row of `table` it selects (embedding, or the pre-multiplied input projection) -- replacing a full pass over the
 * logits + a separate gather per decode step. */
int caphn_gemm_tc_amax(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                       int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, float* amax_val,
                       int* amax_idx, int amax_ld, int* nparts, void* stream);
int caphn_argmax_finish_gather(const float* pval, const int* pidx, int ld, int nparts, long n, const float* table, int E,
                               long long* tok, float* out, long ldo, void* stream);

/* Weights-resident GRU recurrence for a many-style batch (pooled variant; the north star's "keeps each style group's
 * generated W_hh resident in shared memory across timesteps"): rows sorted by style group, cluster i owns the rows of
 * tile i = {first row, rows <= 8, group, 0} and loads THAT group's W_hh slice once for all T steps.  Whh / bhh point at
 * group 0's weights inside Theta [G, theta]; wstride / bstride = theta. */
int caphn_gru_cluster_fwd_grouped(const float* GI, const float* Whh, const float* bhh, float* Hall, float* Hbm,
                                  float* saved, int B, int T, int H, const int* tiles, int ntiles, long wstride,
                                  long bstride, void* stream);
int caphn_gru_cluster_bwd_grouped(const float* dHbm, const float* saved, const float* Hall, const float* Whh, float* dGI,
                                  float* dGH, float* dh0, int B, int T, int H, const int* tiles, int ntiles, long wstride,
                                  void* stream);

/* Cross-entropy forward and gradient operand in ONE pass over the logits (the fused loss nodes; F.cross_entropy +
 * its backward at cc_train_hypernet.py:152-153 / hypernet.py:139-145): caphn_ce_fwd's outputs plus the bf16 hi/lo split of
 * the UNSCALED gradient u = softmax(X) - onehot(tgt) (0 on ignored rows) as a tensor-core operand [M, Vp] (Vp % 64 == 0;
 * lo may be NULL in bf16 mode).  Logits read once, operand written once.  V <= 50000 (the row is staged in shared memory). */
int caphn_ce_fwd_split(const float* X, long ld, const long long* tgt, long M, int V, int has_ignore, long long ignore,
                       float* lse, float* scratch, float* lossbuf, void* hi, void* lo, long Vp, void* stream);
/* caphn_gemm_tc_ex (no ReLU) with a device-side scalar: C = scale_num[0] / max(scale_den[0], 1) * A B^T (+ bias);
 * scale_den may be NULL.  The products that consume caphn_ce_fwd_split's operand pass scale_num = grad_output of the loss
 * and scale_den = lossbuf + 1 (number of valid rows): dH = s * u W_out, [dW_out | db] = s * u^T [H | 1]. */
int caphn_gemm_tc_scaled(const void* Ahi, const void* Alo, long a_ld, int a_mn, const void* Bhi, const void* Blo, long b_ld,
                         int b_mn, long K, float* C, long ldc, const float* bias, int M, int N, int splitk,
                         const float* scale_num, const float* scale_den, void* stream);

/* One greedy-decode step of the pooled captioner (later.py:459-490: argmax feedback -> embedding -> nn.GRUCell) as one
 * launch: finishes the arg-max of the previous vocabulary projection from the partials of caphn_gemm_tc_amax (GI == NULL; the
 * token goes to tok if non-NULL), takes the input projection from row tok of table [V, 3H] (= Emb W_ih^T + b_ih) -- or uses
 * GI [B, 3H] directly (step 0) --, applies the GRU cell with W_hh [3H, H] / b_hh and writes hnew [B, H] plus, if hi != NULL, its
 * bf16 hi / lo operand rows [B, Kp] for the next vocabulary projection.  hnew must not alias hprev.  nparts <= 256
 * (else CAPHN_EINVAL); a row with no candidate in its partials gets token 0. */
int caphn_gru_decode_step(const float* GI, const float* pval, const int* pidx, int ldp, int nparts, const float* table,
                          const float* Whh, const float* bhh, const float* hprev, float* hnew, void* hi, void* lo, long Kp,
                          long long* tok, int B, int H, void* stream);

/* caphn_gru_decode_step with the input token given (beam search: the prev_tok of caphn_beam_step): row b's input projection
 * is row tok[b] of table [V, 3H]; an entry outside [0, V) reads row 0.  No arg-max partials are read, so V is not bounded;
 * the H limits of caphn_gru_decode_step apply.  hnew must not alias hprev. */
int caphn_gru_decode_step_tok(const int* tok, int V, const float* table, const float* Whh, const float* bhh,
                              const float* hprev, float* hnew, void* hi, void* lo, long Kp, int B, int H, void* stream);

/* Weights-resident GRU recurrence without a cluster (csrc/gru_resident.cu): one CTA per 4 batch rows keeps the whole generated
 * W_hh as thread-private weight vectors (shared memory + registers), so every step is CTA-local.  Same contract as
 * caphn_gru_cluster_fwd / _bwd (nn.GRUCell per step + BPTT, later.py:411,418); *ok of the plan call says whether H fits. */
int caphn_gru_resident_plan(int H, int* ok);
int caphn_gru_resident_fwd(const float* GI, const float* Whh, const float* bhh, float* Hall, float* Hbm, float* saved, int B,
                           int T, int H, void* stream);
int caphn_gru_resident_bwd(const float* dHbm, const float* saved, const float* Hall, const float* Whh, float* dGI,
                           float* dGH, float* dh0, int B, int T, int H, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CAPHN_B200_H */
