/* dotaclient_b200 -- C-ABI of the B200-native DotaClient optimizer hot path.
 *
 * The reference (TimZaman/dotaclient @ 8615b90) is pure Python on torch CPU; it has no FFI
 * layer.  Each entry point below replaces a stock-torch/scipy op sequence of the reference's
 * optimizer step and names it (file:line in the reference tree).  A maintainer binds these
 * with ctypes from optimizer.py / policy.py (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer (fp32 unless stated), owned by the caller; nothing is
 *     allocated or freed by the library, nothing is synchronised: work is enqueued on `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - return value: 0 = ok; >0 = cudaError_t; <0 = argument error (DC_EINVAL ...).
 *     dc_last_error() returns a thread-local human-readable message for the last failure.
 *   - bool tensors (masks / actions) are bytes holding 0 or 1 (torch.bool layout).
 *   - "time-major" = [S, B, ...]: token (t, b) lives at row t*B + b.
 *   - compiled for sm_100a only; there is no CPU fallback.
 */
#ifndef DOTACLIENT_B200_H
#define DOTACLIENT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DC_OK 0
#define DC_EINVAL (-1)      /* bad argument */
#define DC_EUNSUPPORTED (-2) /* shape outside what the kernels are built for */

#define DC_CELL_GRU 0  /* gate order r,z,n  (torch.nn.GRU,  policy.py:66) */
#define DC_CELL_LSTM 1 /* gate order i,f,g,o (torch.nn.LSTM; the cell BASELINE.json names) */

#define DC_NUM_HEADS 5    /* enum,x,y,target_unit,ability  (policy.py:46) */
#define DC_LOSS_SLOTS 16  /* layout of the `out` vector of dc_ppo_loss_fwd_bwd, see below */

typedef void *dc_stream_t;

/* Library / device introspection. */
int dc_version(void);
const char *dc_last_error(void);
/* sm count, compute capability of the current device; >0 cudaError_t if there is none. */
int dc_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* ---- GAE -----------------------------------------------------------------------------
 * Replaces advantage_returns()/discount() (optimizer.py:53-64) and the reward reduction that
 * feeds them (optimizer.py:397,417-421) for n_seg rollouts at once.
 *   rewards  [n_rows, n_sub]   sub-rewards per step (n_sub = 10, policy.py:20) or n_sub = 1
 *   values   [n_rows]          critic values (padded steps included, optimizer.py:396)
 *   seg_off  [n_seg+1] int64   rollout r covers rows seg_off[r] .. seg_off[r+1]-1
 *   boot_value [n_seg] or NULL value of the state after the last row   } the trailing elements the
 *   boot_reward[n_seg] or NULL start of the rewards-to-go recursion    } reference appends, both 0
 *                              (NULL = 0: terminated rollouts, optimizer.py:413-420)
 *   adv, ret [n_rows]          outputs
 * deltas in fp32, the two reverse scans accumulate in float64 and round to fp32 exactly like
 * scipy.signal.lfilter + astype(float32) does.  Warp-shuffle segmented scan, one warp / rollout.
 */
int dc_gae_scan(const float *rewards, int n_sub, const float *values, const int64_t *seg_off,
                int n_seg, const float *boot_value, const float *boot_reward, double gamma,
                double lam, float *adv, float *ret, dc_stream_t stream);

/* ---- recurrent core --------------------------------------------------------------------
 * Replaces the time recurrence inside nn.GRU / nn.LSTM (policy.py:66,141) -- forward and
 * backward -- given the input-to-hidden pre-activations of all steps.
 *
 * Forward
 *   gates  [S, B, G, H] in : x_t W_ih^T + b_ih (time-major)      G = 3 (GRU) / 4 (LSTM)
 *                       out: activated gates (r,z,n | i,f,g,o), saved for backward (in place)
 *   w_hh   [G*H, H], b_hh [G*H]   rnn.weight_hh_l0 / rnn.bias_hh_l0
 *   ybuf   [S+1, B, H]  slot 0 = h_0 (in), slot t+1 = h_t (out)   -> y = ybuf[1:], h_n = ybuf[S]
 *   cbuf   [S+1, B, H]  LSTM: slot 0 = c_0 (in), slot t+1 = c_t (out)
 *                       GRU : slot t+1 = W_hn h_{t-1} + b_hn (out, saved for backward)
 *   workspace: dc_rnn_workspace_bytes(cell, B, H) bytes of scratch (W_hh^T for H != 256; at H = 256 the partial-sum
 *              exchange of the cluster backward kernel -- the same buffer serves forward and backward).
 * Kernels by width: H = 128 one-SM weight-resident FFMA2 kernels; H = 256 (the reference's width) 8-CTA-cluster
 * tensor-memory-resident tcgen05 3xTF32 kernels; any other H % 4 == 0 a generic kernel that streams W_hh from L2.
 * Backward (consumes what forward left behind)
 *   gates  in: activated gates   out: dL/d(gates pre-activation wrt the i2h branch) = dgi
 *   cbuf   LSTM: unchanged.  GRU: slot t+1 out = dL/d(W_hn h + b_hn) (the n-gate part of dgh)
 *   dy     [S, B, H]  dL/dy (time-major); dhn/dcn [B, H] or NULL (gradient of the final state)
 *   dh0/dc0 [B, H] or NULL outputs.
 */
size_t dc_rnn_workspace_bytes(int cell, int B, int H);
int dc_rnn_seq_fwd(int cell, float *gates, const float *w_hh, const float *b_hh, float *ybuf,
                   float *cbuf, int B, int S, int H, void *workspace, dc_stream_t stream);
int dc_rnn_seq_bwd(int cell, float *gates, const float *w_hh, const float *ybuf, float *cbuf,
                   const float *dy, const float *dhn, const float *dcn, float *dh0, float *dc0,
                   int B, int S, int H, void *workspace, dc_stream_t stream);

/* ---- fp32-accurate tensor-core GEMM (tcgen05, 3xTF32) ---------------------------------------
 * C[M,N] = A[M,K] * B[N,K]^T (+ bias[N]) (ReLU if relu != 0); row-major fp32 with leading dimensions lda/ldb/ldc.
 * Replaces the library SGEMM of the input-to-hidden projection inside nn.GRU / nn.LSTM (policy.py:66,141:
 * gates = x W_ih^T + b_ih) and of the other 128-aligned dense layers (policy.py:101-126,138).  Each product is
 * evaluated as a_lo*b_hi + a_hi*b_lo + a_hi*b_hi with tf32 hi/lo splits (fp32-level accuracy, ~1e-6 relative).
 * Requirements: N % 128 == 0, K % 32 == 0, 16-byte aligned pointers, ld* % 4 == 0 (dc_gemm_tf32x3_supported).
 */
int dc_gemm_tf32x3_supported(int64_t M, int N, int K);
int dc_gemm_tf32x3(const float *A, int lda, const float *B, int ldb, const float *bias, float *C, int ldc,
                   int64_t M, int N, int K, int relu, dc_stream_t stream);

/* Weight gradient of the same layers: dW[No,Ni] (+)= dY[T,No]^T X[T,Ni], db[No] (+)= column sums of dY (NULL = skip).
 * Replaces the dW/db part of AddmmBackward for those layers (loss.backward(), optimizer.py:672).  Contraction over the
 * token dimension with MN-major tcgen05 operands, split-K over the SMs, deterministic two-stage reduction.
 * Requirements: No % 128 == 0, Ni % 128 == 0; workspace of dc_gemm_wgrad_workspace_bytes(No, Ni) bytes. */
size_t dc_gemm_wgrad_workspace_bytes(int No, int Ni);
int dc_gemm_wgrad_tf32x3(const float *dY, int ldy, const float *X, int ldx, int64_t T, int No, int Ni,
                         float *dW, int ldw, float *db, int accumulate, void *workspace, dc_stream_t stream);

/* Two-level row addressing variants: row r of A / C / dY lives at (r / rows_per_block) * block_stride +
 * (r % rows_per_block) * ld (floats); rows_per_block = 0 selects the plain form.  They let the per-group GEMMs read
 * and write one unit group of the [N, 40, 128] unit-embedding tensor in place, so the torch.cat of policy.py:130-131
 * (and its backward split) never materialises. */
int dc_gemm_tf32x3_blocked(const float *A, int lda, int64_t a_rows_per_block, int64_t a_block_stride,
                           const float *B, int ldb, const float *bias, float *C, int ldc,
                           int64_t c_rows_per_block, int64_t c_block_stride, int64_t M, int N, int K,
                           int relu, dc_stream_t stream);
int dc_gemm_wgrad_tf32x3_blocked(const float *dY, int ldy, int64_t y_rows_per_block, int64_t y_block_stride,
                                 const float *X, int ldx, int64_t T, int No, int Ni, float *dW, int ldw,
                                 float *db, int accumulate, void *workspace, dc_stream_t stream);

/* ---- unit encoder / target-unit head: the bandwidth-bound pieces ------------------------------
 * (policy.py:99-136,144-153; the 128x128 embedding GEMMs themselves are dc_gemm_tf32x3*)
 *   dc_unit_basic_fwd   basic[R,128] = relu(units[R,12] W_b^T + b_b)            policy.py:100,105,...
 *   dc_target_unit_fwd  logits[n,u] = <att[n,:], ue[n,u,:]>, ue = [N,40,128]    policy.py:152-153
 *   dc_target_unit_bwd  d_att[n,:] = sum_u dlogits[n,u] ue[n,u,:];  d_ue[n,u,:] = dlogits[n,u] att[n,:]
 */
int dc_unit_basic_fwd(const float *units, const float *w_b, const float *b_b, float *basic, int64_t R,
                      dc_stream_t stream);
/* The same, also writing the ReLU sign bits of `basic` for dc_unit_dgrad_fused_mask: mask = uint32 [ceil(R/32), 128], bit i of
 * word [b][j] = basic[32b + i][j] > 0, bits of rows >= R are 0.  basic and mask 16-byte aligned. */
int dc_unit_basic_fwd_mask(const float *units, const float *w_b, const float *b_b, float *basic, uint32_t *mask, int64_t R,
                           dc_stream_t stream);
size_t dc_unit_basic_bwd_workspace_bytes(void);   /* partial sums of dW_b / db_b: the workspace of dc_unit_dgrad_fused */
/* Environment encoder (policy.py:55,97): out[n*ld_out + c] = relu(env[n,:3] . W_e[c,:] + b_e[c]), c < 128 -- written into
 * columns [0,128) of the concatenated pre-rnn input row (ld_out = 896), so the reference's torch.cat (policy.py:129-136)
 * is never materialised.  dc_env_bwd: dW_e[128,3] = (d_out * (out>0))^T env, db_e[128] = column sums (deterministic). */
int dc_env_fwd(const float *env, const float *w_e, const float *b_e, float *out, int ld_out, int64_t N,
               dc_stream_t stream);
size_t dc_env_bwd_workspace_bytes(void);
int dc_env_bwd(const float *d_out, const float *out, int ld, const float *env, float *dw_e, float *db_e, int64_t N,
               void *workspace, dc_stream_t stream);
/* Unit-embedding layer with the max-pool fused into the GEMM epilogue (policy.py:101-127): emb = basic[N*n_units,128] W^T is
 * reduced per token to xmax[n*ld_x + c] = max_u emb[n,u,c] + b[c] (also written to xmax_copy when not NULL, policy.py:127) and
 * argmax[n*128 + c] (first maximum wins, like torch.max); the embedding itself is never stored.  n_units = 5 or 16. */
int dc_gemm_unit_max(const float *basic, const float *w, const float *bias, float *xmax, float *xmax_copy, int ld_x,
                     uint8_t *argmax, int64_t n_tokens, int n_units, dc_stream_t stream);
/* Target-unit head without the embedding (policy.py:144-153): logits[n,u] = <q[n, g*128 ..], basic_g[n,u,:]> + q[n, 768+g]
 * with q = att [W_0|...|W_5|b_0..b_5] (ld_q >= 896) and basics[g] = the [N*units_g, 128] basic activations of group g
 * (units 1,5,16,16,1,1).  Backward: s[n, g*128 + j] = sum_u dlogits[n,u] basic_g[n,u,j], s[n, 768+g] = sum_u dlogits[n,u]
 * (zeros in 774..895), so that d_att = s [W_0|...|W_5|b]^T is one GEMM. */
int dc_target_unit_q_fwd(const float *q, int ld_q, const float *const basics[6], float *logits, int64_t N, dc_stream_t stream);
int dc_target_unit_q_bwd(const float *dlogits, const float *const basics[6], float *s, int ld_s, int64_t N, dc_stream_t stream);
/* Backward of one unit-embedding layer WITHOUT the dense [N*units, 128] gradient of the embedding (what the reference's autograd
 * materialises behind policy.py:100-127,152-153).  R[(n,u), c] = (argmax[n*128 + c] == u) ? d_xmax[n*ld_dx + c] (+ d_xmax2[..]) : 0 is
 * the max-pool routing, generated inside the kernels.
 *   dc_unit_wgrad_routed  dW[128,128] = R^T basic,  db[128] = column sums of R            (n_units = 5 or 16; a 1-unit group is
 *                         dc_gemm_wgrad_tf32x3 on d_xmax itself; workspace: dc_gemm_wgrad_workspace_bytes(128, 128))
 *   dc_unit_dgrad_fused   dW_b[128,12] (+)= G^T units, db_b[128] (+)= column sums of G, with
 *                         G[(n,u), j] = (basic[(n,u), j] > 0) * sum_c (R[(n,u), c] + dlogits[n*ld_dl + u] att[n*128 + c]) W[c, j]:
 *                         the whole gradient of the embedding (routing + the target-unit head's rank-1 part) is generated inside
 *                         the kernel; w_t = W^T [128,128]; the ReLU mask is recomputed from units/w_b/b_b (bit-identical to
 *                         dc_unit_basic_fwd); dlogits (already offset to the group's first unit) and att [N,128] are NULL when the
 *                         head was not used; d_xmax NULL = no routing (the enemy-tower layer, policy.py:127).  n_units = 1, 5 or
 *                         16; units, att, d_xmax 16-byte aligned; workspace: dc_unit_basic_bwd_workspace_bytes().
 * The head's share of dW / db is a token-level product (att^T s, s from dc_target_unit_q_bwd) the caller adds. */
int dc_unit_wgrad_routed(const float *d_xmax, const float *d_xmax2, int ld_dx, const uint8_t *argmax, const float *basic,
                         int64_t n_tokens, int n_units, float *dW, float *db, void *workspace, dc_stream_t stream);
int dc_unit_dgrad_fused(const float *d_xmax, const float *d_xmax2, int ld_dx, const uint8_t *argmax, const float *dlogits,
                        int ld_dl, const float *att, const float *w_t, const float *units, const float *w_b,
                        const float *b_b, int64_t n_tokens, int n_units, float *dw_b, float *db_b, int accumulate,
                        void *workspace, dc_stream_t stream);
/* dc_unit_dgrad_fused with the ReLU mask read from the forward pass (dc_unit_basic_fwd_mask of the same rows, 16-byte aligned)
 * instead of recomputed from w_b, b_b: the same results, bit for bit. */
int dc_unit_dgrad_fused_mask(const float *d_xmax, const float *d_xmax2, int ld_dx, const uint8_t *argmax, const float *dlogits,
                             int ld_dl, const float *att, const float *w_t, const float *units, const uint32_t *mask,
                             int64_t n_tokens, int n_units, float *dw_b, float *db_b, int accumulate, void *workspace,
                             dc_stream_t stream);
int dc_target_unit_fwd(const float *att, const float *ue, float *logits, int64_t N, dc_stream_t stream);
int dc_target_unit_bwd(const float *dlogits, const float *att, const float *ue, float *d_att, float *d_ue,
                       int64_t N, dc_stream_t stream);

/* ---- fused PPO loss + gradient ----------------------------------------------------------
 * Replaces optimizer.py:587-589 (advantage normalisation) and :621-665 (masked log-softmax x5,
 * ratio, clipped surrogate, entropy, value loss) AND their autograd backward, for N tokens.
 *   logits[h]  [N, n_h] fp32   n_h = 4,9,9,40,3     masks[h], actions[h] [N, n_h] bytes
 *   old_logp   [N, 5]   log-prob of the taken action per head at prep time (dense form of
 *                       Sequence.log_probs_sel, optimizer.py:387-390); ignored where no action
 *   adv_raw, ret, value [N]
 *   dlogits[h] [N, n_h], dvalue [N]   gradients of the total loss (loss.backward(), :672)
 *   out [DC_LOSS_SLOTS] fp32: 0 loss, 1 policy_loss, 2 entropy_loss, 3 value_loss,
 *       4..8 entropy per head, 9..13 policy loss per head, 14 adv mean, 15 adv std (unbiased)
 *   n_actions [5] int32: rows with a taken action per head (optimizer.py:626,643)
 *   workspace: DC_PPO_WORKSPACE_BYTES of scratch (zeroed by the call itself).
 * Two launches: statistics (counts, advantage mean/std), then loss+grad.
 */
#define DC_PPO_WORKSPACE_BYTES 512
int dc_ppo_loss_fwd_bwd(const float *const logits[DC_NUM_HEADS],
                        const uint8_t *const masks[DC_NUM_HEADS],
                        const uint8_t *const actions[DC_NUM_HEADS], const float *old_logp,
                        const float *adv_raw, const float *ret, const float *value, int64_t N,
                        float e_clip, float entropy_coef, float vf_coef,
                        float *const dlogits[DC_NUM_HEADS], float *dvalue, float *out,
                        int32_t *n_actions, void *workspace, dc_stream_t stream);

/* Same, with row pitches (floats) for logits[h], dlogits[h], value and dvalue: a pitch of 128 lets the four small heads
 * and the value head be column ranges of ONE packed [N,128] tensor-core GEMM output and of its gradient. */
int dc_ppo_loss_fwd_bwd_strided(const float *const logits[DC_NUM_HEADS], const int64_t ld_logits[DC_NUM_HEADS],
                                const uint8_t *const masks[DC_NUM_HEADS],
                                const uint8_t *const actions[DC_NUM_HEADS], const float *old_logp,
                                const float *adv_raw, const float *ret, const float *value, int64_t ld_value,
                                int64_t N, float e_clip, float entropy_coef, float vf_coef,
                                float *const dlogits[DC_NUM_HEADS], const int64_t ld_dlogits[DC_NUM_HEADS],
                                float *dvalue, int64_t ld_dvalue, float *out, int32_t *n_actions,
                                void *workspace, dc_stream_t stream);

/* Log-prob of the taken action per head, [N,5] dense (0 where the head took no action):
 * the no-grad half of experiences_from_rollout (optimizer.py:387-390). */
int dc_selected_logp(const float *const logits[DC_NUM_HEADS],
                     const uint8_t *const masks[DC_NUM_HEADS],
                     const uint8_t *const actions[DC_NUM_HEADS], int64_t N, float *logp_out,
                     dc_stream_t stream);

/* ---- gradient finish: count-divide, grad-norm metrics, clip, Adam ------------------------
 * Replaces distributed.py:57 (grad /= has_grad_count), optimizer.py:674-681 (mean_gradient_norm
 * x2, clip_grad_norm_(0.5), NaN guard, Adam.step) on ONE flat fp32 buffer holding all params.
 *   flat_grad  [total + n_seg]  gradients, followed by n_seg has-grad counts (after the
 *                               all-reduce: number of ranks that had a gradient, distributed.py:36-37)
 *   seg_lo/hi  [n_seg] int64    parameter p covers flat elements seg_lo[p] .. seg_hi[p]-1 (tensors may be padded apart)
 *   seg_head   [n_seg]   int32  -1 = always has a gradient; h>=0 = has one only if head h took
 *                               an action this batch (optimizer.py:627-630: skipped heads leave
 *                               .grad = None, so Adam and the norm mean skip those tensors)
 *   steps      [n_seg]   int32  per-parameter Adam step counters (in/out)
 *   loss_out   the `out` vector of dc_ppo_loss_fwd_bwd (NaN guard, optimizer.py:667,678)
 *   metrics [4] fp32 out: 0 mean grad norm unclipped, 1 clipped, 2 total norm, 3 nan flag (1 =
 *                               NaN seen, parameters left untouched -- the caller raises ValueError)
 * dc_grad_flags writes the local has-grad flags (1/0) into flat_grad[total ..] before the all-reduce.
 */
int dc_grad_flags(float *flat_grad, int64_t total, const int32_t *seg_head, int n_seg,
                  const int32_t *n_actions, dc_stream_t stream);
int dc_grad_finish(float *flat_param, float *flat_grad, float *exp_avg, float *exp_avg_sq,
                   int32_t *steps, const int64_t *seg_lo, const int64_t *seg_hi, const int32_t *seg_head, int n_seg,
                   int64_t total, double lr, double beta1, double beta2, double adam_eps,
                   double max_norm, const float *loss_out, float *metrics, void *workspace,
                   dc_stream_t stream);
#define DC_FINISH_WORKSPACE_BYTES 1024

/* ---- actor side: hierarchical action selection for a batch of A agents in one launch ----------------
 * (policy.py:23-33 MaskedCategorical, :169-178 masked_softmax, :190-216 sample_action/select_actions; caller agent.py:578-674)
 * Heads in DC order (enum 4, x 9, y 9, target_unit 40, ability 3).  logits[h]: A rows with pitch ld[h] floats;
 * masks[h]: [A, n_h] bytes (0/1); u: [A,5] uniforms in [0,1) supplied by the caller (torch.multinomial's RNG stream cannot
 * be reproduced, so the pinned contract is the index function: inverse CDF over the masked probabilities, fp32, sequential
 * in index order -- oracle/ref_policy.py:sample_index).  chosen[A,5]: enum first, then x,y (enum 1) / target_unit (2) /
 * ability (3); -1 for heads that were not sampled.  logp[A,5] (nullable): log-probability of each chosen entry. */
int dc_select_actions(const float *const logits[DC_NUM_HEADS], const int64_t ld[DC_NUM_HEADS],
                      const uint8_t *const masks[DC_NUM_HEADS], const float *u, int64_t A, int32_t *chosen,
                      float *logp, dc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DOTACLIENT_B200_H */
