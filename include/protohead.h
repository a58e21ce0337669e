/*
 * protohead.h -- C ABI of libprotohead_b200.so: ProtoPFormer's prototype head on B200 (sm_100a).
 *
 * The reference (zju-vipa/ProtoPFormer) has no FFI for this path: it is a Python nn.Module whose arithmetic is
 * ~35 ATen library calls (protopformer.py:141-335).  This library is what a maintainer binds instead of those
 * calls (ctypes stub in INTEGRATION.md; the shipped binding is protopformer_b200/_lib.py).  Each entry point
 * cites the reference lines it replaces.
 *
 * Conventions (all entry points):
 *   - extern "C", plain pointers and ints; every pointer is a DEVICE pointer owned and pre-allocated by the
 *     caller unless the parameter comment says "host".
 *   - `stream` is a cudaStream_t passed as void*.  Nothing allocates, nothing synchronises, no global state
 *     except a per-thread last-error string -> every call is CUDA-graph capturable.
 *   - return 0 on success, a negative PPH_E* argument error, or a positive cudaError_t from the launch.
 *     pph_last_error_string() describes the last non-zero return on the calling thread.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns a cudaError_t.
 *   - float tensors are fp32 row-major contiguous; "bf16" is the 16-bit brain float (uint16_t storage).
 *
 * Symbols (B images, N patch tokens, K reserved tokens, Din backbone width, D prototype dim, P local
 * prototypes, Pg global prototypes, C classes, m = P / C prototypes per class):
 */
#ifndef PROTOHEAD_B200_H
#define PROTOHEAD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPH_VERSION 202

/* argument errors */
#define PPH_EINVAL   (-1)   /* bad dimension / null pointer */
#define PPH_EUNSUP   (-2)   /* shape outside what the sm_100a kernels were built for */
#define PPH_EDRIVER  (-3)   /* cuTensorMapEncodeTiled unavailable / failed */

/* similarity precision modes (pph_similarity_fwd `mode`) */
#define PPH_MODE_FP32_FMA 0  /* CUDA-core FP32 FMA contraction (exact-order reference mode, materialises maps) */
#define PPH_MODE_BF16X3   1  /* tcgen05 bf16 tensor cores, 3-term split operands (hi*hi + hi*lo + lo*hi), fp32-grade */
#define PPH_MODE_BF16     2  /* tcgen05 bf16 tensor cores, single pass */

/* prototype activation function, protopformer.py:228-234 */
#define PPH_ACT_LOG    0     /* log((d+1)/(d+eps)) */
#define PPH_ACT_LINEAR 1     /* -d */

typedef void* pph_stream_t;  /* cudaStream_t */

int         pph_version(void);
const char* pph_last_error_string(void);
/* number of SMs of the current device (persistent-grid sizing), or <0 */
int         pph_sm_count(void);
/* Variant / measurement switches (process-wide; the library itself never reads the environment):
 *   "pdl" 0|1 programmatic dependent launch on every kernel; "sim_lanes" n, "sim_shared" 0|1, "sim_epi" 0|1: tcgen05
 *   similarity CTA plan / epilogue variants; "rollout" 1|2|3 and "classmap" 1|2: kernel versions of those rows.
 * Returns 0, or PPH_EINVAL for an unknown name. */
int         pph_set_option(const char* name, int value);

/* (a1) protopformer.py:157-158  topk(cls_token_attn, K)[1].sort()[0]
 * scores [B,H,N] (H>=1; H>1: the mean over H is taken first), idx32 [B,K] ascending, idx64 [B,K] or NULL.
 * N <= 1024, 1 <= K <= N.  Ties: the lower token index wins. */
int pph_select_topk(const float* scores, int B, int H, int N, int K,
                    int32_t* idx32, int64_t* idx64, pph_stream_t stream);

/* (a2) protopformer.py:159-172 + ctor :109-113  gather -> 1x1 conv ('regular' add-on) -> sigmoid, for the K
 * selected patch tokens and the CLS token of every image.
 * tokens [B,1+N,Din], idx32 [B,K], Wa [D,Din], ba [D] ->
 *   Zs [B,K,D] fp32, Zc [B,D] fp32, z2s [B,K] = |Zs|^2, z2c [B] = |Zc|^2,
 * and the tensor-core operands, taken from the CENTRED features z' = z - center (the squared distance is
 * translation invariant; centring sigmoid outputs at 0.5 keeps the tcgen05 accumulator ~40x smaller, which is what
 * makes its truncating fp32 accumulation meet the 1e-4 bar):
 *   Zs_hi/Zs_lo [B*K,D] bf16 split (hi = rn(z'), lo = rn(z' - hi)), Zc_hi/Zc_lo [B,D],
 *   z2s_ctr [B,K] / z2c_ctr [B] = |z'|^2 (fp32; the norms PPH_MODE_BF16X3 must be given),
 *   z2s_hi  [B,K] / z2c_hi  [B] = |hi|^2 (norms of the ROUNDED operand; the norms PPH_MODE_BF16 must be given).
 * The eight tensor-core-side outputs may be NULL. */
int pph_addon_fwd(const float* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                  int B, int N, int Din, int D, int K,
                  float* Zs, float* Zc, float* z2s, float* z2c,
                  float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                  uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo, pph_stream_t stream);

/* operand preparation for the tensor-core modes: V [R,D] fp32 -> v2 [R] = |V|^2 (the p2 term of
 * protopformer.py:207-208) and, from v' = v - center: hi/lo bf16 split [R,D], v2_ctr [R] = |v'|^2, v2_hi [R] = |hi|^2.
 * `center` must equal the one given to pph_addon_fwd.  Any output may be NULL. */
int pph_split_rows(const float* V, int R, int D, float center, uint16_t* hi, uint16_t* lo, float* v2, float* v2_ctr,
                   float* v2_hi, pph_stream_t stream);

/* (a3,a4,a5) protopformer.py:201-218, 228-234, 236-247  squared-L2 distances of every selected token to every
 * local prototype (and of the CLS token to every global prototype), log/linear similarity, max over tokens.
 * Local:  dmin_l [B,P] = min_k relu(z2 - 2 z.p + p2), argmin_l [B,P] (token slot 0..K-1, lowest on ties),
 *         act_l [B,P] = act(dmin_l).      Global: dmin_g [B,Pg], act_g [B,Pg].
 * mode FP32_FMA reads Zs/Zc/Pl/Pg (fp32) and can also write the materialised maps dist_map / act_map [B,P,K]
 * (protopformer.py:301 aux `distances`, :344 `proto_acts`); the tcgen05 modes read the centred bf16 operands and
 * want z2s/z2c/p2l/p2g = the matching norms (PPH_MODE_BF16X3: the *_ctr norms; PPH_MODE_BF16: the *_hi norms, lo
 * pointers unused), never write the maps (dist_map/act_map must be NULL) and require D % 64 == 0, 64 <= D <= 512,
 * 1 <= K <= 256. */
int pph_similarity_fwd(int mode, int act_fn, float eps, int B, int K, int D, int P, int Pg,
                       const float* Zs, const float* Zc, const float* z2s, const float* z2c,
                       const uint16_t* Zs_hi, const uint16_t* Zs_lo, const uint16_t* Zc_hi, const uint16_t* Zc_lo,
                       const float* Pl, const float* Pgl, const float* p2l, const float* p2g,
                       const uint16_t* Pl_hi, const uint16_t* Pl_lo, const uint16_t* Pg_hi, const uint16_t* Pg_lo,
                       float* dmin_l, int32_t* argmin_l, float* act_l, float* dmin_g, float* act_g,
                       float* dist_map, float* act_map, pph_stream_t stream);

/* Host-side introspection of the tensor-core launch plan for a shape (no device access, no launch): which kernel
 * (resident-prototype v2 or streaming v1), grid, image-group walkers per prototype tile, pipeline stages, global chunk.
 * out (host int[16]) = {v2, grid, lanes, n_local_ctas, stages, b_tile_bytes, smem_bytes, global_chunk, MT_l, NG_l, MT_g,
 * NB_g, images_per_tile, umma_n_local, umma_n_global, n_tiles}; coverage (host, optional, n_tiles ints, caller-zeroed):
 * incremented once per visit of tile (local: group*MT_l + mt; global: n_local + chunk*MT_g + mt) by the CTA/job walk
 * the kernels perform -- the CPU test suite checks that every entry ends at exactly 1.  sms <= 0: 148. */
int pph_similarity_plan(int mode, int B, int K, int D, int P, int Pg, int sms, int* out /* host */,
                        int* coverage /* host */);

/* (a6) protopformer.py:297-300 / 314-316  logits = gc * act_g Wg^T + (1-gc) * act_l Wl^T
 * Wl [C,P], Wg [C,Pg] -> logits, logits_g, logits_l [B,C] */
int pph_logits_fwd(const float* act_l, const float* act_g, const float* Wl, const float* Wg,
                   int B, int P, int Pg, int C, float global_coe,
                   float* logits, float* logits_g, float* logits_l, pph_stream_t stream);

/* (a7) protopformer.py:249-288  PPC loss.  For image b and its label y the m prototypes y*m..y*m+m-1:
 * activation rows over the K selected tokens are recomputed from Zs/Pl in fp32 (the reference gathers them
 * from the (B,P,K) map), placed on the side x side grid by idx32, -> weighted mean / variance -> the two losses.
 * labels [B] int64.  Saved for backward: dslice [B,m,K] (distances), stats [B,m,8] = S, mu_r, mu_c, V_r, V_c, pre_cov, 0, 0.
 * losses [2] = (ppc_cov_loss, ppc_mean_loss); partial [B,2] and counter [1] (uint32, zero before first use,
 * self-resetting) are scratch for the deterministic final sum. */
int pph_ppc_fwd(const float* Zs, const float* z2s, const float* Pl, const float* p2l,
                const int32_t* idx32, const int64_t* labels,
                int B, int K, int D, int P, int m, int N, int act_fn, float eps,
                float cov_thresh, float mean_thresh,
                float* dslice, float* stats, float* partial, uint32_t* counter, float* losses, pph_stream_t stream);

/* backward of pph_ppc_fwd.  Upstream gradients of (cov, mean): g_losses[2] (device, may be NULL = 1) multiplied by
 * the host scalars g_scale_cov / g_scale_mean (e.g. the loss coefficients of engine_proto.py:61-64).
 * accumulate = 0: dZs [B,K,D] is OVERWRITTEN with the PPC contribution and dP [P,D] must be zero-filled by the
 * caller (rows of shared labels are added atomically).  accumulate = 1: the contribution is ADDED to dZs / dP that
 * already hold the similarity gradients (fused training step: no extra buffers, no extra add kernels). */
int pph_ppc_bwd(const float* Zs, const float* Pl, const int32_t* idx32, const int64_t* labels,
                const float* dslice, const float* stats, const float* g_losses,
                float g_scale_cov, float g_scale_mean,
                int B, int K, int D, int P, int m, int N, int act_fn, float eps,
                float cov_thresh, float mean_thresh, int accumulate,
                float* dZs, float* dP, pph_stream_t stream);

/* (a8, part 1) autograd of protopformer.py:297-300 and :228-244 collapsed to one scalar per (b,p):
 *   g_l[b,p] = (1-gc) * (sum_c dlogits[b,c] Wl[c,p] [+ gc_extra terms]) * act'(dmin_l[b,p]) * [dmin_l > 0]
 *   g_g[b,p] = gc * (sum_c dlogits[b,c] Wg[c,p]) * act'(dmin_g[b,p]) * [dmin_g > 0]
 * dlogits, dlogits_g, dlogits_l [B,C] (the latter two may be NULL: no upstream gradient on logits_global/local). */
int pph_logits_bwd(const float* dlogits, const float* dlogits_g, const float* dlogits_l,
                   const float* Wl, const float* Wg, const float* dmin_l, const float* dmin_g,
                   int B, int P, int Pg, int C, float global_coe, int act_fn, float eps,
                   float* g_l, float* g_g, pph_stream_t stream);

/* Weight gradients of the last layers, for callers that unfreeze them (the reference freezes them, protopformer.py:130-131,
 * but its autograd would train them once `requires_grad` is set; main.py:370 then averages them with the rest): the
 * derivative of protopformer.py:297-300 / 314-316 w.r.t. Wl and Wg,
 *   dWl[c,p] = sum_b ((1-gc) dlogits[b,c] + dlogits_l[b,c]) act_l[b,p]      dWg[c,p] = sum_b (gc dlogits[b,c] + dlogits_g[b,c]) act_g[b,p]
 * dlogits [B,C] (upstream gradient of the combined logits), dlogits_g / dlogits_l [B,C] or NULL (no upstream gradient on
 * logits_global / logits_local), act_l [B,P], act_g [B,Pg] (pph_similarity_fwd).  dWl [C,P], dWg [C,Pg] are OVERWRITTEN;
 * either may be NULL (not computed).  Every entry is one fixed-order sum over b (no atomics: bit-reproducible); the kernel
 * never waits on another CTA, so it may share the device with the step's co-resident kernels.  B, P, C >= 1; no bound on C. */
int pph_last_layer_wgrad(const float* dlogits, const float* dlogits_g, const float* dlogits_l,
                         const float* act_l, const float* act_g, int B, int P, int Pg, int C, float global_coe,
                         float* dWl, float* dWg, pph_stream_t stream);

/* (a8, part 2) max-pool routing + distance backward (SURVEY.md 8(d)(iv)):
 *   dPl[p,:]   = 2 * sum_b g_l[b,p] * (Pl[p,:] - Zs[b,argmin[b,p],:])      dPg[p,:] = 2 * sum_b g_g[b,p] * (Pg[p,:] - Zc[b,:])
 *   dZs[b,k,:] = 2 * sum_{p: argmin[b,p]=k} g_l[b,p] * (Zs[b,k,:] - Pl[p,:])   dZc[b,:] = 2 * sum_p g_g[b,p] * (Zc[b,:] - Pg[p,:])
 * All four outputs are OVERWRITTEN; every row is summed in a fixed order (bit-reproducible).
 * `workspace`: caller-owned device scratch of pph_similarity_bwd_ws_bytes() bytes, ZERO-FILLED once before its
 * first use (it holds the token bins and self-resetting counters).
 * `parts`: PPH_BWD_BIN (bin the prototypes by argmin token; needs only argmin_l + workspace, so it can run on another
 * stream as soon as the forward similarity is done) | PPH_BWD_GRADS (the four gradients; requires the bins).
 * add_dZs [B,K,D] / add_dPl [P,D] (either may be NULL): gradients from elsewhere (the PPC loss) that are added while
 * dZs / dPl are written, so that they can be produced concurrently and cost no extra pass. */
#define PPH_BWD_BIN   1
#define PPH_BWD_GRADS 2
int pph_similarity_bwd_ws_bytes(int B, int K, int D, int P, int Pg, long long* bytes /* host */);
int pph_similarity_bwd(const float* g_l, const float* g_g, const int32_t* argmin_l,
                       const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                       int B, int K, int D, int P, int Pg, void* workspace, int parts,
                       const float* add_dZs, const float* add_dPl,
                       float* dZs, float* dZc, float* dPl, float* dPg, pph_stream_t stream);

/* (a8, part 3) backward of pph_addon_fwd: dpre = dZ * Z * (1-Z);  dWa = dpre^T X_sel;  dba = sum dpre;
 * dtokens[b, 1+idx] = dpre Wa (CLS row 0 likewise), every other row zero.
 * dWa [D,Din], dba [D], dtokens [B,1+N,Din] are OVERWRITTEN (dtokens may be NULL: no gradient to the backbone).
 * `workspace`: caller-owned device scratch of pph_addon_bwd_ws_bytes() bytes (split-K partials of the weight
 * gradient, summed in a fixed order).
 * `parts`: PPH_ADDON_WGRAD (dWa, dba) | PPH_ADDON_DGRAD (dtokens); the two are independent and may be issued on
 * different streams. */
#define PPH_ADDON_WGRAD 1
#define PPH_ADDON_DGRAD 2
int pph_addon_bwd_ws_bytes(int B, int N, int Din, int D, int K, long long* bytes /* host */);
int pph_addon_bwd(const float* tokens, const int32_t* idx32, const float* Wa,
                  const float* Zs, const float* Zc, const float* dZs, const float* dZc,
                  int B, int N, int Din, int D, int K, void* workspace, int parts,
                  float* dWa, float* dba, float* dtokens, pph_stream_t stream);

/* loss tail adjacent to the head (engine_proto.py:51, 61-64): ce = CrossEntropy(logits, labels) (mean over B),
 * out_losses[4] = (ce + cov_coe*ppc[0] + mean_coe*ppc[1], ce, ppc[0], ppc[1]) and
 * dlogits [B,C] = (softmax - onehot) / B * upstream   (NULL: forward only).  ppc_losses [2] may be NULL (= 0).
 * partial [B] and counter [1] (zero before first use, self-resetting) are scratch. */
int pph_loss_tail(const float* logits, const int64_t* labels, const float* ppc_losses,
                  float cov_coe, float mean_coe, float upstream, int B, int C,
                  float* partial, uint32_t* counter, float* out_losses, float* dlogits, pph_stream_t stream);

/* out_losses[4] = (ce + cov_coe*ppc[0] + mean_coe*ppc[1], ce, ppc[0], ppc[1]) from ce_losses[4] = the out_losses of a
 * pph_loss_tail call made with ppc_losses = NULL (engine_proto.py:61-64).  Splitting the sum off lets the cross-entropy
 * gradient start before the PPC loss (computed on another stream) is available.  ppc_losses may be NULL (= 0). */
int pph_loss_combine(const float* ce_losses, const float* ppc_losses, float cov_coe, float mean_coe,
                     float* out_losses, pph_stream_t stream);

/* (next #1, producer of the selection score) tools/deit_models_attn.py:99-124 attn_rollout + :226
 * `cls_token_attn = attn_rollout(all_attn)[:, 0, 1:]`, computed without forming the (T,T) products:
 *   per layer l and image b: fused = head_fusion over H of attn_l[b] (T x T); the k_discard smallest entries of the
 *   flattened map are zeroed (k_discard = int(T*T*discard_ratio), computed by the caller exactly as the reference does;
 *   ties at the threshold: lowest flat index first); a_l = rownorm((fused + identity_w * I) / (1 + identity_w));
 *   v = v0[b] (or e_0 when v0 is NULL); for l = L-1 .. 0: v <- v a_l;   scores[b] = v[drop_first:].
 * attn_layers: HOST array of L DEVICE pointers, each a contiguous fp32 [B,H,T,T] tensor (they are copied into the kernel
 * arguments: nothing is retained).  head_fusion: 0 mean, 1 max, 2 min.  identity_w = 0.2 in the reference.
 * v0 [B,T] optional start row (CaiT, cait_models_attn.py:255-259); drop_first = 1 drops the CLS column (DeiT).
 * scores [B, T - drop_first].  workspace: pph_rollout_ws_bytes() bytes of device scratch (sparse per-layer matrices).
 * Fused selection (north_star (a): score reduction + per-image top-k in one pass): K > 0 also writes the ascending
 * index list of the K largest scores of each image, idx32 [B,K] (and idx64 [B,K] unless NULL), exactly what
 * pph_select_topk would return on `scores` (protopformer.py:157-158, deit_models_attn.py:229-230); K = 0: scores only.
 * L <= 32, 2 <= T <= 224. */
#define PPH_FUSE_MEAN 0
#define PPH_FUSE_MAX  1
#define PPH_FUSE_MIN  2
int pph_rollout_ws_bytes(int L, int B, int T, int k_discard, long long* bytes /* host */);
int pph_rollout_scores(const float* const* attn_layers /* host array of device pointers */, int L, int B, int H, int T,
                       int k_discard, int head_fusion, float identity_w, const float* v0, int drop_first,
                       void* workspace, float* scores, int K, int32_t* idx32, int64_t* idx64, pph_stream_t stream);

/* (next #3, optimizer tail) torch.optim.AdamW as the reference builds it for the head's parameter groups
 * (tools/create_optimizer.py:31-39, :92; engine_proto.py:76-78), all tensors in ONE launch:
 *   p *= 1 - lr*wd;  m += (1-b1)(g - m);  v = b2 v + (1-b2) g g;  p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * n_seg <= 8 tensors: params / grads / exp_avg / exp_avg_sq are HOST arrays of DEVICE pointers (fp32, numel[i] elements,
 * copied into the kernel arguments); group[i] (host) selects the tensor's row of hyper.
 * hyper: DEVICE [8][2] = (lr, weight_decay) per parameter group -- device memory so that a CUDA graph holding this
 * launch follows the lr schedule.  step_state: DEVICE int[2] = {t, ticket}: t = updates done so far (0 before the
 * first call), incremented by the kernel; ticket must be 0.  grads are multiplied by grad_scale first (loss scaling /
 * sum-reduced gradients). */
int pph_adamw_step(int n_seg, float* const* params, const float* const* grads, float* const* exp_avg,
                   float* const* exp_avg_sq, const long long* numel /* host */, const int* group /* host */,
                   const float* hyper, double beta1, double beta2, float eps, float grad_scale,
                   int* step_state, pph_stream_t stream);

/* CaiT start row for pph_rollout_scores (tools/cait_models_attn.py:223-259): the n_cls class-attention maps
 * cls_layers[c] = [B,H,1,Tc] (host array of device pointers) are fused over heads, their k_discard = int(Tc*ratio)
 * smallest entries zeroed (ties: lowest index first), identity_w added on the CLS column (`I[:1]`), rows normalised;
 * v0 [B, Tc-1] = mean over the n_cls rows without the CLS column.  Then
 * pph_rollout_scores(patch_layers, ..., T = Tc-1, v0, drop_first = 0) = `cls_attn_ma[:, 0]` (cait_models_attn.py:328-330). */
int pph_rollout_cls_rows(const float* const* cls_layers /* host array of device pointers */, int n_cls, int B, int H,
                         int Tc, int k_discard, int head_fusion, float identity_w, float* v0, pph_stream_t stream);

/* (next #4, consumers of the materialised map) eval_interpretability.py:195-225 / main_visualize.py:343-388:
 * activation maps of the m prototypes of each image's label on the ORIGINAL side x side token grid, zeros on pruned
 * tokens: maps[b, q, idx32[b,k]] = act(relu(z2s[b,k] + (p2l[p] - 2 Zs[b,k].Pl[p]))), p = labels[b]*m + q.
 * Zs [B,K,D], z2s [B,K] (= |Zs|^2, from pph_addon_fwd), Pl [P,D], p2l [P] (from pph_split_rows), labels [B] int64,
 * maps [B,m,N] fully OVERWRITTEN.  The (B,P,K) map is never formed. */
int pph_class_maps(const float* Zs, const float* z2s, const float* Pl, const float* p2l,
                   const int32_t* idx32, const int64_t* labels, int B, int K, int D, int P, int m, int N,
                   int act_fn, float eps, float* maps, pph_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Fused training / inference step (round 2): the same path in FIVE launches
 *   pph_head_prep -> pph_similarity_fwd -> pph_head_mid -> pph_similarity_bwd2 -> pph_addon_bwd2
 * (tools/engine_proto.py:49-76 for the head: forward, cross-entropy, PPC loss, backward).  The modular entry points
 * above remain the operator-level API (autograd functions of the drop-in PPNet) and the fallback for shapes these
 * kernels were not built for (every *_supported() below answers on the host, without a device).
 * ------------------------------------------------------------------------------------------------------------------ */

/* (a1)+(a2)+operand preparation in one launch: pph_select_topk (NaN scores rank first, as torch.topk) -> pph_addon_fwd
 * for scores [B,H,N], tokens [B,1+N,Din]; plus pph_split_rows of Pl [P,D] and Pgl [Pg,D] (either may be NULL / 0 rows).
 * Outputs as documented at those entry points; idx64 and all bf16 / *_ctr / *_hi outputs may be NULL. */
int pph_head_prep_supported(int B, int N, int Din, int D, int K);
int pph_head_prep(const float* scores, const float* tokens, const float* Wa, const float* ba,
                  int B, int H, int N, int Din, int D, int K, float center,
                  int32_t* idx32, int64_t* idx64,
                  float* Zs, float* Zc, float* z2s, float* z2c, float* z2s_ctr, float* z2c_ctr,
                  float* z2s_hi, float* z2c_hi, uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                  const float* Pl, int P, uint16_t* Pl_hi, uint16_t* Pl_lo, float* p2l, float* p2l_ctr, float* p2l_hi,
                  const float* Pgl, int Pg, uint16_t* Pg_hi, uint16_t* Pg_lo, float* p2g, float* p2g_ctr, float* p2g_hi,
                  pph_stream_t stream);

/* (a6) + loss tail + (a8 part 1) [+ token bins of (a8 part 2)] [+ (a7) PPC loss forward and backward] in one launch:
 *   logits / logits_g / logits_l [B,C] as pph_logits_fwd; losses[4] = (ce + cov_coe*cov + mean_coe*mean, ce, cov, mean) as
 *   pph_loss_tail + pph_loss_combine (cov = mean = 0 when use_ppc = 0); and, when train != 0:
 *   dlogits [B,C]; g_l [B,P], g_g [B,Pg] as pph_logits_bwd (no upstream gradient on logits_global/local);
 *   pairT [(P+Pg)][Bp][2] fp32, Bp = B rounded up to 64: (g, bit pattern of the int32 token slot) per (prototype, image),
 *   token slot K (= the CLS row) for global prototypes, zeros for images >= B (pairT may be NULL: only
 *   pph_similarity_bwd2 reads it);
 *   the token bins (and, with use_ppc, the images sorted by class) of pph_similarity_bwd2 in bwd_workspace;
 *   with use_ppc: dZs_ppc [B,K,D] = d(cov_coe*cov + mean_coe*mean)*upstream / dZs (OVERWRITTEN) and
 *   dP_img [B,m,D] = the same gradient w.r.t. the m label-class prototype rows, per image (summed over the images of a
 *   class by pph_similarity_bwd2 in image order: deterministic).
 * use_ppc: 0 no PPC loss | 1 PPC role inside this launch | 2 this launch runs everything but the PPC role and a second,
 * concurrent call with use_ppc = 3 (same arguments, another stream) runs only that role: whichever finishes second
 * writes losses[0] -- lets the PPC loss overlap the last layers instead of lengthening the launch.  Adding 4 to use_ppc
 * makes dZs_ppc leave as the pre-activation gradient (times Z (1 - Z)): the form pph_addon_bwd3's dpre_add_s takes.
 * workspace: pph_head_mid_ws_bytes() bytes, ZERO-FILLED once before first use (grid-barrier and ticket counters, all
 * self-resetting).  C <= 256; B <= 64 * (SM count / 2).  Out-of-range labels are clamped.
 * When pph_last_layer_pattern, run on the same workspace before this call, found both Wl and Wg in the class-connection
 * pattern, the last layers take their class-sum form (O(B P) instead of O(B P C), same results up to summation order);
 * otherwise the general product.  The launch clears the verdicts it used: each call needs a check of its own. */
int pph_head_mid_ws_bytes(int B, int K, int D, int P, int Pg, int C, int m, long long* bytes /* host */);
int pph_head_mid(const float* act_l, const float* act_g, const float* dmin_l, const float* dmin_g,
                 const int32_t* argmin_l, const float* Wl, const float* Wg, const int64_t* labels,
                 int B, int K, int D, int P, int Pg, int C, int m, int N,
                 float global_coe, int act_fn, float eps, float upstream, int train,
                 int use_ppc, const float* Zs, const float* z2s, const float* Pl, const float* p2l,
                 const int32_t* idx32, float cov_thresh, float mean_thresh, float cov_coe, float mean_coe,
                 void* workspace, void* bwd_workspace,
                 float* logits, float* logits_g, float* logits_l, float* losses, float* dlogits,
                 float* g_l, float* g_g, float* pairT, float* dZs_ppc, float* dP_img,
                 float* losses_mirror /* NULL, or 4 floats (16-byte aligned; may be mapped pinned HOST memory) that receive
                                         (total, ce, ppc_cov, ppc_mean) with the same store that completes losses[0]: the
                                         caller's device->host read of the step result without a copy node */,
                 pph_stream_t stream);

/* Device-side check of the last layers Wl [C,P] and Wg [C,Pg] (Wg may be NULL when Pg = 0) against the pattern of
 * PPNet.set_last_layer_incorrect_connection (protopformer.py:367-386): with m = n / C, W[c,p] == a where p / m == c and
 * == b elsewhere, a = W[0,0], b = W[1,0] (b = a when C = 1), by exact float equality; n % C != 0 fails.  Writes its
 * verdicts into the first PPH_LL_PATTERN_BYTES of `workspace` (a pph_head_mid workspace) for the pph_head_mid call that
 * follows on the stream: two records {int32 ok; float a; float b; int32 unused}, Wl then Wg (Pg = 0: ok, a = b = 0).
 * One launch, integer atomics only, no host synchronisation -- meant to run inside the captured step, every step. */
#define PPH_LL_PATTERN_BYTES 32
int pph_last_layer_pattern(const float* Wl, int P, const float* Wg, int Pg, int C, void* workspace, pph_stream_t stream);

/* (a8 part 2), second implementation: same results as pph_similarity_bwd(PPH_BWD_GRADS) from operands staged in shared
 * memory by feature slices (no L2 row gathers), every row summed in a fixed order (no atomics on data).  Three kernels,
 * selected by `parts`, independent of each other -- meant for concurrent streams:
 *   PPH_BWD2_TOKENS -> dZs [B,K,D]     PPH_BWD2_PROTOS -> dPl [P,D], dPg [Pg,D]     PPH_BWD2_CLS -> dZc [B,D]
 * g_l / g_g / pairT and the bins + class lists in bwd_workspace come from pph_head_mid (same launch sequence).
 * add_dZs [B,K,D] (or NULL) is added to dZs; dP_img [B,m,D] (or NULL) is added to the label-class rows of dPl, summed
 * over the images of a class in image order.  dpre_out != 0: dZs / dZc are multiplied by Z (1 - Z) while they are
 * written, i.e. they hold the pre-activation gradient pph_addon_bwd2 consumes.
 * bwd_workspace: pph_similarity_bwd2_ws_bytes() bytes, ZERO-FILLED once before first use.  D % 16 == 0. */
#define PPH_BWD2_TOKENS 1
#define PPH_BWD2_PROTOS 2
#define PPH_BWD2_CLS    4
int pph_similarity_bwd2_supported(int B, int K, int D, int P, int Pg);
int pph_similarity_bwd2_ws_bytes(int B, int K, int D, int P, long long* bytes /* host */);
int pph_similarity_bwd2(int parts, const float* g_l, const float* g_g, const float* pairT, void* bwd_workspace,
                        const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                        int B, int K, int D, int P, int Pg, int m,
                        const float* add_dZs, const float* dP_img, int dpre_out,
                        float* dZs, float* dZc, float* dPl, float* dPg, pph_stream_t stream);

/* pph_similarity_bwd(PPH_BWD_GRADS) inside the fused step: the argmin-routed gather kernel of round 1 fed by the bins
 * and class lists pph_head_mid left in `step_workspace` (= the bwd_workspace given to it); `workspace` is a
 * pph_similarity_bwd_ws_bytes() scratch (zero-filled once).  add_dZs / dP_img / dpre_out as pph_similarity_bwd2. */
int pph_similarity_bwd_fused(int parts /* 1 token-side rows | 2 prototype rows; or 4 alone: dPl += PPC rows of dP_img */,
                             const float* g_l, const float* g_g, const int32_t* argmin_l,
                             const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                             int B, int K, int D, int P, int Pg, int m, void* workspace, void* step_workspace,
                             const float* add_dZs, const float* dP_img, int dpre_out,
                             float* dZs, float* dZc, float* dPl, float* dPg, pph_stream_t stream);

/* (a8 part 3), second implementation: backward of pph_addon_fwd from the PRE-ACTIVATION gradient
 * dpre = dZ * Z * (1 - Z) (dpre_s [B,K,D] for the selected tokens, dpre_c [B,D] for the CLS token), exact FP32,
 * deterministic.  parts: PPH_ADDON_WGRAD -> dWa [D,Din], dba [D]; PPH_ADDON_DGRAD -> dtokens [B,1+N,Din] (every row
 * written: zeros for tokens that were not selected).  workspace: pph_addon_bwd2_ws_bytes() bytes, ZERO-FILLED once
 * before first use.  Din % 8 == 0, D % 4 == 0. */
int pph_addon_bwd2_supported(int B, int N, int Din, int D, int K);
int pph_addon_bwd2_ws_bytes(int B, int N, int Din, int D, int K, long long* bytes /* host */);
int pph_addon_bwd2(int parts, const float* tokens, const int32_t* idx32, const float* Wa,
                   const float* dpre_s, const float* dpre_c,
                   int B, int N, int Din, int D, int K, void* workspace,
                   float* dWa, float* dba, float* dtokens, pph_stream_t stream);

/* The add-on layer products on the single-shot tcgen05 kernel (one 128 x BN output tile per CTA, its whole k range
 * resident in shared memory, 3-term bf16 split as pph_addon_fwd):
 *   pph_addon_fwd2 = pph_addon_fwd (same outputs, same numerics) with the output columns split over CTAs;
 *   pph_addon_bwd3 = pph_addon_bwd2 (inputs dpre_s / dpre_c) on tensor cores; with PPH_ADDON_DGRAD the rows of dtokens
 *   that belong to selected tokens (and the CLS rows) are written, every other row must have been ZERO-FILLED by the
 *   caller; PPH_ADDON_WGRAD reduces its split-k partials in-kernel behind a grid barrier (needs <= SM-count CTAs).
 * pph_addon_tc2_supported: bit 0 forward, bit 1 DGRAD, bit 2 WGRAD, bit 3 pph_select_addon_fwd can run this shape.  workspace:
 * pph_addon_tc2_ws_bytes() bytes, ZERO-FILLED once before first use (shared by the three calls of a step). */
int pph_addon_tc2_supported(int B, int N, int Din, int D, int K);
int pph_addon_tc2_ws_bytes(int B, int N, int Din, int D, int K, long long* bytes /* host */);
int pph_addon_fwd2(const float* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                   int B, int N, int Din, int D, int K,
                   float* Zs, float* Zc, float* z2s, float* z2c,
                   float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                   uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                   void* workspace, pph_stream_t stream);
/* Selection + gather + add-on in ONE launch (protopformer.py:157-172): pph_select_topk's ranking (same total order, head
 * mean over H, NaN first) runs in the prologue of pph_addon_fwd2's kernel -- every CTA ranks the scores of the images its
 * row tile touches -- and idx32 [B,K] is an OUTPUT.  Same numerics as pph_select_topk followed by pph_addon_fwd2. */
int pph_select_addon_fwd(const float* scores /* [B,H,N] */, int H, const float* tokens, const float* Wa, const float* ba,
                         int B, int N, int Din, int D, int K, int32_t* idx32 /* out */,
                         float* Zs, float* Zc, float* z2s, float* z2c,
                         float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                         uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                         void* workspace, pph_stream_t stream);
int pph_addon_bwd3(int parts, const float* tokens, const int32_t* idx32, const float* Wa,
                   const float* dpre_s, const float* dpre_c, const float* dpre_add_s /* [B,K,D] added to dpre_s, or NULL */,
                   int B, int N, int Din, int D, int K, void* workspace,
                   float* dWa, float* dba, float* dtokens, pph_stream_t stream);

/* PPC loss on a DENSE activation map: `get_PPC_loss(total_proto_act, cls_attn_rollout, original_fea_len, label)` as the
 * reference writes it (protopformer.py:259-288) for callers that hold the (B,P,h,w) map as a tensor.  act [B,P,K] (the map
 * flattened over h,w), idx32 [B,K] ascending selected tokens (pph_select_topk of cls_attn_rollout, :273-274), labels [B].
 * fwd: losses[0] = L_cov, losses[1] = L_mean; stats [B,m,8], partial [B,2] and a ZERO-INITIALISED counter are scratch kept for
 * the backward.  bwd: dact [B,P,K] is written completely (zeros outside the label-class rows) for the upstream scalars
 * g_cov, g_mean (device pointers).  1 <= m <= 32, N a perfect square.  Deterministic. */
int pph_ppc_dense_fwd(const float* act, const int32_t* idx32, const int64_t* labels, int B, int P, int K, int m, int N,
                      float cov_thresh, float mean_thresh, float* stats, float* partial, unsigned int* counter,
                      float* losses, pph_stream_t stream);
int pph_ppc_dense_bwd(const float* act, const int32_t* idx32, const int64_t* labels, const float* stats,
                      const float* g_cov, const float* g_mean, int B, int P, int K, int m, int N, float mean_thresh,
                      float* dact, pph_stream_t stream);

/* Selection-first input transfer for tokens that live in pinned (mapped) HOST memory: copies the CLS row and the K
 * selected token rows of every image (idx32 from pph_select_topk, protopformer.py:156-166) from tokens_host
 * [B, 1+N, Din] to the same positions of tokens_dev [B, 1+N, Din] by zero-copy loads over PCIe; the other rows of
 * tokens_dev are left untouched (the head's forward and backward never read them).  tokens_host must be page-locked
 * host memory (cudaHostAlloc / cudaHostRegister); PPH_EINVAL otherwise.  Din a multiple of 4. */
int pph_gather_rows_host(const float* tokens_host, const int32_t* idx32, int B, int N, int Din, int K,
                         float* tokens_dev, int n_ctas, pph_stream_t stream);

/* Gradient exchange of the data-parallel head (reference: DistributedDataParallel, main.py:369-371) as ONE kernel over
 * NVLink / NVSwitch peer memory: averages buf[lo, lo + n) IN PLACE over `world` ranks.  buf_ptrs (HOST array, `world`
 * entries) holds the address of the same peer-mapped ("symmetric") buffer on every rank as mapped into this process
 * (entry `rank` is the local one); multicast_ptr is the NVLS multicast mapping of that buffer or 0 (then rank r sums
 * chunk r of every peer in rank order and stores the average into every peer; with multicast the switch does both:
 * multimem.ld_reduce / multimem.st).  A flag block of pph_peer_flag_bytes() bytes, ZERO-FILLED once before the first call
 * and followed by a barrier over the ranks, lives inside every rank's buffer at flag_offset_bytes (16-byte aligned, behind
 * the data).  Every rank must issue the same sequence of calls per `slot` (0..3; calls that may overlap in time use
 * different slots) with the same lo, n, n_ctas.  lo and n are multiples of 4 floats.  Safe to record in CUDA graphs
 * (flags are monotonically increasing epochs).  A peer that never arrives traps the kernel instead of hanging. */
int pph_peer_flag_bytes(long long* bytes /* host */);
int pph_peer_allreduce(const unsigned long long* buf_ptrs /* host */, unsigned long long multicast_ptr,
                       long long flag_offset_bytes, int rank, int world, long long lo, long long n,
                       int n_ctas, int slot, pph_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PROTOHEAD_B200_H */
