/* ups_b200 — C ABI of the B200-native part-disentanglement hot path.
 *
 * The reference (CompVis/unsupervised-part-segmentation) has no FFI: its boundary for this
 * path is the set of Python helper signatures in {cub,pennaction,deepfashion}/code.  Each
 * entry point below replaces the TensorFlow op chain behind one of those helpers; the
 * Python package `ups_b200` binds them with ctypes and re-exposes the reference's
 * signatures (see INTEGRATION.md).  Citations are relative to the reference checkout.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to a contiguous fp32 buffer unless stated; NHWC;
 *     `P` = H*W pixels per sample; labels are int64 (tf.argmax's dtype)
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it:
 *     no allocation, no free, no synchronisation, no host-visible side effect
 *   - scratch memory is caller-owned: ask ups_workspace_bytes() and pass `ws`
 *   - return value: 0 on success, negative UPS_E_* otherwise; ups_last_error_string()
 *     (thread-local) describes the last failure.  Nothing throws.
 *   - re-entrant and thread-safe: no global mutable state besides the thread-local error
 */
#ifndef UPS_B200_H
#define UPS_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UPS_OK 0
#define UPS_E_INVALID (-1)   /* bad shape / null pointer / unsupported size */
#define UPS_E_CUDA (-2)      /* a CUDA runtime call or launch failed */
#define UPS_E_WORKSPACE (-3) /* workspace too small */

const char* ups_version(void);
const char* ups_last_error_string(void);
/* ups_version(): "ups_b200 <version> (sm_100a, src=<hash>)"; <hash> = first 12 hex digits of the SHA-256 over the sources
 * and headers the binary was built from (unsupervised-part-segmentation_b200/build.py::source_hash), so that a binary
 * that does not correspond to the sources beside it is detected and rebuilt.
 * ups_launch_count(): number of kernels this library has launched on the calling thread since the last reset
 * (thread-local diagnostics counter, bench.py's `gpu_launches`). */
long long ups_launch_count(void);
void ups_launch_count_reset(void);

/* ---- workspace sizes --------------------------------------------------------------- */
enum ups_op {
    UPS_OP_TPS_SOLVE = 0,   /* none */
    UPS_OP_POOL = 1,        /* part_pool_fwd / encode_fwd partial sums */
    UPS_OP_INJECT_BWD = 2,  /* part_inject_bwd / decode_bwd dfeat partial sums */
    UPS_OP_POOL_BWD = 3,    /* none */
    UPS_OP_STEP = 4,        /* ups_step_* (max over the four fused calls and their unfused stand-ins) */
    UPS_OP_MOMENTS = 5,     /* ups_mask_moments_fwd partial sums */
    UPS_OP_KL = 6,          /* ups_categorical_kl_fwd partial sums */
    UPS_OP_MUMFORD_SHAH = 7, /* ups_mumford_shah_fwd partial sums (only when `sums` is requested) */
    UPS_OP_LOGIT_PRIORS = 8, /* ups_logit_priors_fwd partial sums */
    UPS_OP_WEAK_XENT = 9    /* ups_weak_xent_fwd partial sums (P = pixels per sample, B*P pixels in total) */
};
size_t ups_workspace_bytes(int op, int B, int P, int K, int F);

/* ---- image ingest ------------------------------------------------------------------- */
/* The normalisation the reference's data pipeline applies on the host right before the views are fed
 * (cub/code/data/data.py:134,152; pennaction/code/data/data.py:134,152):
 *     o.astype(np.float32) * 2.0 / 255.0 - 1.0
 * src: n uint8 values (any NHWC image batch), dst: n fp32 values; both 16-byte aligned device pointers.
 * Bit-identical to the numpy expression (fp32 multiply, correctly rounded divide, subtract). */
int ups_views_u8_to_f32(const unsigned char* src, float* dst, long long n, void* stream);
/* The other direction of the host boundary: int64 part labels (tf.argmax's dtype, cub/code/SB_model48i/model.py:447,470)
 * narrowed to one byte per pixel for the read-back of the label map (n_parts <= 255; the evaluation code only uses the
 * labels as an index map, cub/code/eval/eval_iclr_01/eval_01.py:237-239).  labels 16-byte aligned, out 4-byte aligned. */
int ups_labels_i64_to_u8(const long long* labels, unsigned char* out, long long n, void* stream);

/* ---- thin-plate-spline warp -------------------------------------------------------- */
/* make_input_tps_param(tps_param) — baselines/unsupervised-disentangling/transformations.py:59-77
 * coord,vector [N,8,2]; offset,offset_2 [N,1,2]; t_scal [N,2]; rot_mat [N,2,2] -> t_vector [N,8,2]
 * (the returned `coord` is the input coord unchanged). */
int ups_tps_input_param(const float* coord, const float* vector, const float* offset, const float* offset_2,
                        const float* t_scal, const float* rot_mat, float* t_vector, int N, void* stream);
/* ThinPlateSpline._solve_system — transformations.py:215-235 (incl. the ::-1 flip of :95-96)
 * coord, vector [N,8,2] as passed to ThinPlateSpline -> T [N,2,11]. */
int ups_tps_solve(const float* coord, const float* vector, float* T, int N, void* stream);
/* ThinPlateSpline(U, coord, vector, out_size, n_c, move, scal) — transformations.py:93-244
 * (_meshgrid :171-188, _transform :190-213, _interpolate :114-169).
 * U [N,H,W,C]; coord [N,8,2]; T [N,2,11] from ups_tps_solve; move [N,1,2] / scal [N,2] or both NULL;
 * out [N,out_h,out_w,C]; mesh [N,out_h,out_w,2] = (y, x) or NULL. */
int ups_tps_warp_fwd(const float* U, const float* coord, const float* T, const float* move, const float* scal,
                     float* out, float* mesh, int N, int H, int W, int C, int out_h, int out_w, void* stream);
/* gradient of ups_tps_warp_fwd w.r.t. U (4-way scatter-add; floor/clip carry no gradient).
 * dU [N,H,W,C] is zero-filled by the call. */
int ups_tps_warp_bwd(const float* g_out, const float* coord, const float* T, const float* move, const float* scal,
                     float* dU, int N, int H, int W, int C, int out_h, int out_w, void* stream);

/* TrainModel.make_tps — cub/code/SB_model48i/model.py:298-310: view0 and view0_target are warped with
 * the SAME parameters.  The pair calls warp U [N,...] and, for the first N2 samples, a second image
 * set U2 [N2,...] at the same sample positions (the radial-basis grid is evaluated once). */
int ups_tps_warp_pair_fwd(const float* U, const float* U2, const float* coord, const float* T, float* out, float* out2,
                          int N, int N2, int H, int W, int C, int out_h, int out_w, void* stream);
int ups_tps_warp_pair_bwd(const float* g_out, const float* g_out2, const float* coord, const float* T, float* dU,
                          float* dU2, int N, int N2, int H, int W, int C, int out_h, int out_w, void* stream);

/* ---- part-map softmax / hard max / straight-through / argmax ------------------------ */
/* nn.softmax(x, spatial=False) — cub/code/nn.py:58-62, fused with the consumers at
 * cub/code/SB_model48i/model.py:426-473: probs, optional int64 argmax labels (first index),
 * optional straight_through_estimator(hard_max(probs,3), probs).  logits [n_pix,K]. */
int ups_part_softmax_fwd(const float* logits, float* probs, long long* labels, float* hard_st, long long n_pix,
                         int K, void* stream);
/* dx = p*(g - sum_j g_j p_j)  (TF SoftmaxGrad) */
int ups_part_softmax_bwd(const float* probs, const float* g, float* dlogits, long long n_pix, int K, void* stream);
/* same with up to three cotangents summed inside the kernel ((g + g2) + g3; g2, g3 may be NULL) */
int ups_part_softmax_bwd2(const float* probs, const float* g, const float* g2, const float* g3, float* dlogits,
                          long long n_pix, int K, void* stream);
/* elementwise sums of the unfused step: y += a*x ; out[v] = (g_views ? g_views[v] : 0) + (v == idx ? extra : 0)
 * for V views of n_per_view floats (the cotangent of the warped views: model.py:282-311 differentiated) */
int ups_axpy(const float* x, float* y, long long n, float a, void* stream);
int ups_views_cotangent(const float* g_views, const float* extra, float* out, int V, int idx, long long n_per_view,
                        void* stream);
/* nn.spatial_softmax — cub/code/nn.py:65-71: softmax over the P axis for every (n, c); x [N,P,C]. */
int ups_spatial_softmax_fwd(const float* x, float* probs, int N, int P, int C, void* stream);
int ups_spatial_softmax_bwd(const float* probs, const float* g, float* dx, int N, int P, int C, void* stream);
/* nn.hard_max(y, axis=last) — cub/code/nn.py:134-136 (every tied maximum gets 1.0) */
int ups_hard_max_fwd(const float* y, float* out, long long n_pix, int K, void* stream);
/* nn.straight_through_estimator(y_hard, y) forward value fl(fl(y_hard-y)+y) — cub/code/nn.py:154-168 */
int ups_straight_through_fwd(const float* y_hard, const float* y, float* out, long long n, void* stream);
/* tf.argmax(y, 3) — cub/code/SB_model48i/model.py:447,465,470 ; nn.mask2hotmask nn.py:2086-2089 */
int ups_argmax_fwd(const float* y, long long* labels, long long n_pix, int K, void* stream);
int ups_one_hot_fwd(const long long* labels, float* out, long long n_pix, int K, void* stream);

/* ---- mask_parts / apply_partwise ---------------------------------------------------- */
/* mask_parts(image, mask) — cub/code/SB_model48i/model.py:176-187.
 * image [B,P,C], mask [B,P,K] -> parts.  part_major=0: [B,P,K,C] (the reference's layout);
 * part_major=1: [K*B,P,C] with row k*B+b, i.e. already folded as nn.apply_partwise does
 * (cub/code/nn.py:100-103). */
int ups_mask_parts_fwd(const float* image, const float* mask, float* parts, int B, int P, int K, int C,
                       int part_major, void* stream);
/* dimage[b,p,c] = sum_k g*mask ; dmask[b,p,k] = sum_c g*image ; either output may be NULL */
int ups_mask_parts_bwd(const float* g_parts, const float* image, const float* mask, float* dimage, float* dmask,
                       int B, int P, int K, int C, int part_major, void* stream);
/* the two transposes of nn.apply_partwise — cub/code/nn.py:100-103 and :108-112.
 * fold: x [B,P,K,C] -> y [K*B,P,C];  unfold: y [K*B,P,C] -> x [B,P,K,C]. */
int ups_partwise_fold(const float* x, float* y, int B, int P, int K, int C, void* stream);
int ups_partwise_unfold(const float* y, float* x, int B, int P, int K, int C, void* stream);

/* ---- mask-weighted pooling ---------------------------------------------------------- */
/* grouped=1: pool_features(feature_map, mask) — deepfashion/code/foo.py:287-307
 *            fmap [B,P,K*Fg], out[b,k,f] = scale * sum_p fmap[b,p,k*Fg+f]*mask[b,p,k]  (scale = 1/P)
 * grouped=0: get_features(features, part_map, slim=True) — baselines/unsupervised-disentangling/ops.py:182-193
 *            fmap [B,P,Fg],   out[b,k,f] = scale * sum_p fmap[b,p,f]*mask[b,p,k]
 * out [B,K,Fg]; ws from ups_workspace_bytes(UPS_OP_POOL, B, P, K, Fg). */
int ups_part_pool_fwd(const float* fmap, const float* mask, float* out, int B, int P, int K, int Fg, int grouped,
                      float scale, void* ws, size_t ws_bytes, void* stream);
/* dfmap / dmask may be NULL */
int ups_part_pool_bwd(const float* g_out, const float* fmap, const float* mask, float* dfmap, float* dmask, int B,
                      int P, int K, int Fg, int grouped, float scale, void* stream);

/* ---- unpooling / projection onto the part maps ---------------------------------------- */
/* unpool_features(feature_vectors, mask) — cub/code/SB_model48i/model.py:225-249,
 * deepfashion/code/foo.py:462-498: out[b,p,k,f] = mask[b,p,k]*feat[b,k,f]  ([B,P,K,F]). */
int ups_part_unpool_fwd(const float* feat, const float* mask, float* out, int B, int P, int K, int F, void* stream);
int ups_part_unpool_bwd(const float* g_out, const float* feat, const float* mask, float* dfeat, float* dmask, int B,
                        int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
/* reduce_sum(unpool_features(feat, mask), 3) ++ mask — cub/code/SB_model48i/model.py:482-484,
 * without the [B,P,K,F] intermediate: inj [B,P,F+K]. */
int ups_part_inject_fwd(const float* feat, const float* mask, float* inj, int B, int P, int K, int F, void* stream);
/* dmask[b,p,k] = sum_f g[b,p,f]*feat[b,k,f] + g[b,p,F+k] ; dfeat[b,k,f] = sum_p mask[b,p,k]*g[b,p,f] */
int ups_part_inject_bwd(const float* g_inj, const float* feat, const float* mask, float* dfeat, float* dmask, int B,
                        int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
/* nn.unpool_features_gathered(feature_vectors, labels) — cub/code/nn.py:2469-2487: out [B,P,F] */
int ups_part_gather_fwd(const float* feat, const long long* labels, float* out, int B, int P, int K, int F,
                        void* stream);

/* ---- the fused per-step path (SURVEY.md 8d: K2..K5; K1/K6 are the TPS calls above) --------
 * encode side (view 1): m1 = softmax(l1); mh = ST(hard_max(m1)); parts = mask_parts(img1, mh)
 *   written part-major [K*B,P,3]; pooled[b,k,c] = mean_p mh*img1   — model.py:429,453-455,478, :50-52 */
int ups_step_encode_fwd(const float* l1, const float* img1, float* m1, float* parts_pm, float* pooled, int B, int P,
                        int K, void* ws, size_t ws_bytes, void* stream);
/* decode side (view 0): m0 = softmax(l0); labels0 = argmax(m0); mh = ST(hard_max(m0));
 *   inj = sum_k unpool(feat, mh) ++ mh   — model.py:426,434-436,447,482-484 */
int ups_step_decode_fwd(const float* l0, const float* feat, float* m0, long long* labels0, float* inj, int B, int P,
                        int K, int F, void* stream);
/* backward of the decode side: dl0 = softmax_bwd(m0, inject_bwd_dmask(g_inj) + g_m0), dfeat.
 * g_m0 (cotangent arriving at the probabilities from the losses) may be NULL. */
int ups_step_decode_bwd(const float* g_inj, const float* m0, const float* g_m0, const float* feat, float* dl0,
                        float* dfeat, int B, int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
/* Same contract as ups_step_decode_bwd as a persistent TMA + tcgen05 pipeline: the (P x F).(F x K)
 * contraction on the tensor cores (kind::tf32, 3xTF32 split, fp32 accumulation in TMEM), dfeat as a
 * deterministic scatter-add.  Needs K in {16,32}, F == 64, P % 128 == 0, B*P < 2^31.
 * ws from ups_workspace_bytes(UPS_OP_STEP, ...) (holds the per-chunk dfeat partials and the chunk counter). */
int ups_step_decode_bwd_tc(const float* g_inj, const float* m0, const float* g_m0, const float* feat, float* dl0,
                           float* dfeat, int B, int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
/* backward of the encode side: dm1 = sum_c img1*(g_parts + g_pooled/P); dl1 = softmax_bwd(m1, dm1 + g_m1);
 * dimg1 (optional) = sum_k mh*(g_parts + g_pooled/P).  g_pooled, g_m1, dimg1 may be NULL. */
int ups_step_encode_bwd(const float* g_parts_pm, const float* g_pooled, const float* img1, const float* m1,
                        const float* g_m1, float* dl1, float* dimg1, int B, int P, int K, void* stream);

/* ---- mask statistics on the probabilities (SURVEY.md 8f: N1, N2) --------------------------
 * probs_to_mu_sigma(probs, scaling_factor) — cub/code/nn.py:1541-1587 (call sites
 * cub/code/SB_model48i/model.py:440,458,689).  probs [B,H,W,K]; scaling [B,K];
 * mu [B,K,2] = (y, x) on the linspace(-1,1) grid; sigma [B,K,2,2]; moments [B,K,5] = the raw sums
 * (p*y, p*x, p*y*y, p*y*x, p*x*x) kept for the backward.  ws from ups_workspace_bytes(UPS_OP_MOMENTS, B, H*W, K, 0). */
int ups_mask_moments_fwd(const float* probs, const float* scaling, float* mu, float* sigma, float* moments, int B,
                         int H, int W, int K, void* ws, size_t ws_bytes, void* stream);
/* dprobs [B,H,W,K] from g_mu [B,K,2] / g_sigma [B,K,2,2] (either may be NULL); scaling_factor gets no gradient
 * (the reference always passes a constant). */
int ups_mask_moments_bwd(const float* g_mu, const float* g_sigma, const float* scaling, const float* moments,
                         float* dprobs, int B, int H, int W, int K, void* stream);
/* categorical_kl(probs) — cub/code/SB_model48i/model.py:21-25: mean over pixels of sum_k p*log(K*p + 1e-20).
 * probs [n_pix,K] -> out[1].  ws from ups_workspace_bytes(UPS_OP_KL, ...). */
int ups_categorical_kl_fwd(const float* probs, float* out, long long n_pix, int K, void* ws, size_t ws_bytes,
                           void* stream);
int ups_categorical_kl_bwd(const float* probs, const float* g_out, float* dprobs, long long n_pix, int K, void* stream);

/* ---- mask priors and mean-field sampling around the softmax (SURVEY.md 8f N2/N3) ------------------ */
/* mumford_shah(x, alpha, lambda_) / edge_set(x, alpha, lambda_) — cub/code/nn.py:1357-1392 (finite differences
 * fd_kernel/tf_grad/tf_squared_grad :1357-1378), call site cub/code/SB_model48i/model.py:744-769.
 * x [B,H,W,K] -> r, smooth, contour, edges [B,H,W,K] (each may be NULL) and sums [B,4,K] = sum over (h,w) of
 * (r, smooth, contour, x) (may be NULL; these are what the training step squares).  Elementwise outputs are
 * bit-identical to the reference expression.  ws from ups_workspace_bytes(UPS_OP_MUMFORD_SHAH, B, H*W, K, 0),
 * needed only with `sums`. */
int ups_mumford_shah_fwd(const float* x, float alpha, float lambda, float* r, float* smooth, float* contour,
                         float* edges, float* sums, int B, int H, int W, int K, void* ws, size_t ws_bytes, void* stream);
/* dx [B,H,W,K] from elementwise cotangents g_r / g_smooth / g_contour [B,H,W,K] and/or g_sums [B,4,K] (each may be
 * NULL); tf.minimum routes the gradient to alpha*g where alpha*g <= lambda, tf.where to the selected branch. */
int ups_mumford_shah_bwd(const float* x, float alpha, float lambda, const float* g_r, const float* g_smooth,
                         const float* g_contour, const float* g_sums, float* dx, int B, int H, int W, int K, void* stream);
/* MeanFieldDistribution.kl / kl_improper_gmrf / kl_tv — cub/code/nn.py:1429-1451 (call site model.py:1071):
 * mean [B,H,W,K] -> out[3] = (0.5*sum mean^2, 0.5*sum (dy^2+dx^2), sum |dy|+|dx|), each averaged over the batch;
 * dy/dx = tf.image.image_gradients (forward differences, zero in the last row / column).
 * ws from ups_workspace_bytes(UPS_OP_LOGIT_PRIORS, ...). */
int ups_logit_priors_fwd(const float* mean, float* out, int B, int H, int W, int K, void* ws, size_t ws_bytes, void* stream);
/* dmean [B,H,W,K] = sum_i g_out[i] * d out[i] / d mean, g_out[3] on the device. */
int ups_logit_priors_bwd(const float* mean, const float* g_out, float* dmean, int B, int H, int W, int K, void* stream);
/* MeanFieldDistribution.sample(noise_level) — cub/code/nn.py:1421-1427 (call site model.py:420-421):
 * out = mean + noise_level*eps, n elements; the N(0,1) draw `eps` is an input.  ups_part_softmax_sampled_fwd fuses
 * this in front of the softmax. */
int ups_mean_field_sample_fwd(const float* mean, const float* eps, float noise_level, float* out, long long n, void* stream);
/* softmax(MeanFieldDistribution.sample()) in one pass: like ups_part_softmax_fwd on logits = mean + noise_level*eps;
 * logits_out (may be NULL) receives the sampled logits (model.py:423-424 keeps them as m0_logits / m1_logits). */
int ups_part_softmax_sampled_fwd(const float* mean, const float* eps, float noise_level, float* logits_out, float* probs,
                                 int64_t* labels, float* hard, long long n_pix, int K, void* stream);
/* weak cross entropy — cub/code/SB_model48i/model.py:667-681: mean over pixels of
 * softmax_cross_entropy_with_logits_v2(labels, logits) with labels = ST(hard_max(softmax(logits))) (mode 0,
 * entropy_func "cross_entropy") or softmax(logits) (mode 1, "entropy").  logits [n_pix,K] -> out[1].
 * ws from ups_workspace_bytes(UPS_OP_WEAK_XENT, B, P, K, 0) with B*P = n_pix. */
int ups_weak_xent_fwd(const float* logits, int mode, float* out, long long n_pix, int K, void* ws, size_t ws_bytes,
                      void* stream);
/* dlogits with TF's registered gradient of the v2 op (into logits and into labels, the latter chained through the
 * straight-through estimator and the softmax). */
int ups_weak_xent_bwd(const float* logits, int mode, const float* g_out, float* dlogits, long long n_pix, int K,
                      void* stream);
/* mask2rgb(mask, make_hot) — cub/code/nn.py:2067-2083 (mask2hotmask :2086-2089; eval_01.py:276-281):
 * mask [n_pix,K], table [K,3] = (colors - 0.5)*2 (prepared by the caller as the reference does in numpy) ->
 * out [n_pix,3]; make_hot: colour of the first maximum, else sum_k mask_k*table_k. */
int ups_mask2rgb_fwd(const float* mask, const float* table, int make_hot, float* out, long long n_pix, int K, void* stream);

/* ---- the decoder's first convolution on the part assignment (SURVEY.md 8f N4) ----------------------
 * Replaces   injected = tf.concat([tf.reduce_sum(unpool_features(feat, mask), 3), mask], 3)   cub/code/SB_model48i/model.py:482-484
 *            h = nn.conv2d(injected, config[0])  (3x3, stride 1, SAME, + bias)               model.py:96 (`dd`, :485), cub/code/nn.py:617-664
 * without materialising `injected` [B,h,w,F+K]:  h = b + conv3x3(mask, G[b])  with the per-sample filter table
 *   G[b,t,k,o] = sum_f feat[b,k,f] V[t,f,o] + V[t,F+k,o],   t = 3*i + j,  V = TensorFlow HWIO [3,3,F+K,Co].
 * K <= 32, Co a multiple of 4 in [4,128]. */
/* feat [B,K,F], V [9,F+K,Co] -> G [B,9,K,Co] */
int ups_inject_conv_table_fwd(const float* feat, const float* V, float* G, int B, int K, int F, int Co, void* stream);
/* dG [B,9,K,Co] -> dfeat [B,K,F] (may be NULL), dV [9,F+K,Co] (may be NULL; summed over the batch) */
int ups_inject_conv_table_bwd(const float* dG, const float* feat, const float* V, float* dfeat, float* dV, int B, int K,
                              int F, int Co, void* stream);
/* mask [B,H,W,K] (any values; the straight-through hard mask of model.py:473 takes the one-non-zero fast path),
 * G [B,9,K,Co], bias [Co] -> out [B,H,W,Co] */
int ups_inject_conv_fwd(const float* mask, const float* G, const float* bias, float* out, int B, int H, int W, int K,
                        int Co, void* stream);
/* g_out [B,H,W,Co] -> dmask [B,H,W,K], dG [B,9,K,Co], db [Co] (may be NULL).
 * probs != NULL: the mask is ST(hard_max(probs)) of probs = softmax(logits) (nn.py:117-168); dmask (+ g_extra, the
 * cotangent reaching the probabilities from elsewhere, may be NULL) is passed through the straight-through estimator
 * and the softmax backward, and `dmask` receives dlogits instead.
 * ws from ups_inject_conv_workspace_bytes (per-split partial sums, reduced in a fixed order: deterministic). */
int ups_inject_conv_bwd(const float* g_out, const float* mask, const float* G, const float* probs, const float* g_extra,
                        float* dmask, float* dG, float* db, int B, int H, int W, int K, int Co, void* ws, size_t ws_bytes,
                        void* stream);
size_t ups_inject_conv_workspace_bytes(int B, int H, int W, int K, int Co);
/* host-only query of the backward tiling: out6 = (variant: 0 does not fit / 1 CUDA cores / 2 mma.sync, tile rows, CTAs per
 * sample, tiles per CTA, dynamic shared memory bytes per CTA, tiles per sample).  No device work. */
int ups_inject_conv_bwd_plan(int B, int H, int W, int K, int Co, int* out6);

/* ---- the appearance encoder's first convolution on the masked part images (SURVEY.md 8f N4, encoder side) ----
 * Replaces   view1_parts = mask_parts(view1, encoding_mask)                      cub/code/SB_model48i/model.py:176-187, :478
 *            nn.apply_partwise(view1_parts, e_alpha) -> fold to [K*B,h,w,3]       cub/code/nn.py:81-113
 *            e_alpha's first layer nn.conv2d(x, config[0]) (3x3, SAME, + bias)    model.py:40, cub/code/nn.py:617-664
 * without materialising the part images: img [B,H,W,3], mask [B,H,W,K], V [9,3,Co] (HWIO flattened), bias [Co]
 * -> out_pm [K*B,H,W,Co] part-major (row k*B+b, the batch layout apply_partwise hands the encoder).
 */
int ups_parts_conv_fwd(const float* img, const float* mask, const float* V, const float* bias, float* out_pm, int B,
                       int H, int W, int K, int C, int Co, void* stream);
/* backward: g_out_pm [K*B,H,W,Co] -> dmask [B,H,W,K] (the cotangent of the encoding mask), dV [9,3,Co] (may be NULL),
 * db [Co] (may be NULL).  probs != NULL: the mask is ST(hard_max(probs)); dmask (+ g_extra, the cotangent reaching the
 * probabilities from elsewhere, may be NULL) goes through the straight-through estimator and the softmax backward and
 * `dmask` receives dlogits.  The image gets no gradient (the reference's inputs are placeholders,
 * cub/code/SB_model48i/model.py:316-327).  Co in {8,16,32,64}.
 * ws from ups_parts_conv_bwd_workspace_bytes (plane-major dmask staging + partial sums reduced in a fixed order). */
int ups_parts_conv_bwd(const float* g_out_pm, const float* img, const float* mask, const float* V, const float* probs,
                       const float* g_extra, float* dmask, float* dV, float* db, int B, int H, int W, int K, int C, int Co,
                       void* ws, size_t ws_bytes, void* stream);
size_t ups_parts_conv_bwd_workspace_bytes(int B, int H, int W, int K, int Co);

/* tfutils.draw_rect(mu, patch_size, patch_size, [h, w, 1]) — cub/code/SB_model48i/model.py:442 (the patch masks around
 * the part centres; `tfutils` is not vendored in the reference tree, so the convention is this library's and is stated
 * here): centers [N,2] int32 = (row, column) in pixels; out [N,H,W] = 1 on rows [cy - ph/2, cy - ph/2 + ph) x columns
 * [cx - pw/2, cx - pw/2 + pw) clipped to the image, 0 elsewhere.  No gradient (the call site stops it, model.py:441,449). */
int ups_draw_rect_fwd(const int* centers, float* out, int N, int ph, int pw, int H, int W, void* stream);

/* Part counts that are not a power of two (the reference ships n_parts = 25, train_cub_subset_tps.yaml:132) run on the
 * fused kernels of the next power of two Kp: the [.,K] tensors are padded to [.,Kp] rows (logits with -inf: exp_canon
 * gives exactly 0 and the canonical pair-tree sum is defined on the zero-padded terms, so probabilities, masks and
 * labels are bit-identical), results are cut back to K.  ups_copy_rows is that row copy: dst[r, 0:n_cols] = src[r, 0:n_cols],
 * dst[r, n_cols:n_cols+n_fill] = fill (strides in floats).  The *_planes variants of the encode-side kernels take the
 * number of part planes that really exist in parts / g_parts (Kpl <= K): padding planes are neither written nor read. */
int ups_copy_rows(const float* src, long long src_stride, float* dst, long long dst_stride, long long n_rows, int n_cols,
                  int n_fill, float fill, void* stream);
int ups_step_encode_fwd_planes(const float* l1, const float* img1, float* m1, float* parts_pm, float* pooled, int B, int P,
                               int K, int Kpl, void* ws, size_t ws_bytes, void* stream);
int ups_step_encode_bwd_planes(const float* g_parts_pm, const float* g_pooled, const float* img1, const float* m1,
                               const float* g_m1, float* dl1, float* dimg1, int B, int P, int K, int Kpl, void* stream);

/* ups_tps_warp_pair_bwd with the cotangent formed on the fly: sample b of the N warped samples receives
 * g_out[b] (zeros when g_out is NULL) + extra[b - x0] for b in [x0, x0 + xn); g_out2 / dU2 as in the pair variant (may be
 * NULL).  The fused step uses it to add the encode side's cotangent of warped view 1 (dimg1) to the caller's g_warped
 * without materialising the sum; samples whose cotangent is identically zero are skipped. */
int ups_tps_warp_bwd_sum(const float* g_out, const float* g_out2, const float* extra, int x0, int xn, const float* coord,
                         const float* T, float* dU, float* dU2, int N, int N2, int H, int W, int C, int out_h, int out_w,
                         void* stream);

/* The same kernels with an explicit ROW LENGTH (in floats) for the one [.,K]-shaped input each of them can read in place when
 * K is a padded part count: l0 (decode forward), l1 (encode forward), g_m0 (decode backward), g_m1 (encode backward).
 * row == K is the ordinary call; row < K (e.g. 25 for K = 32) reads the caller's contiguous [., row] tensor element-wise
 * (parts >= row are -inf for logits, 0 for cotangents) and saves the padded copy.  All other tensors keep K-float rows. */
int ups_step_decode_fwd_rows(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0, float* inj, int B,
                             int P, int K, int F, void* stream);
int ups_step_encode_fwd_rows(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm, float* pooled, int B,
                             int P, int K, int Kpl, void* ws, size_t ws_bytes, void* stream);
int ups_step_decode_bwd_rows(const float* g_inj, const float* m0, const float* g_m0, int gm_row, const float* feat, float* dl0,
                             float* dfeat, int B, int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
int ups_step_decode_bwd_tc_rows(const float* g_inj, const float* m0, const float* g_m0, int gm_row, const float* feat,
                                float* dl0, float* dfeat, int B, int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
int ups_step_encode_bwd_rows(const float* g_parts_pm, const float* g_pooled, const float* img1, const float* m1,
                             const float* g_m1, int gm_row, float* dl1, float* dimg1, int B, int P, int K, int Kpl,
                             void* stream);
int ups_step_warp_decode_fwd_rows(const float* U, const float* U2, const float* coord, const float* T, float* out, float* out2,
                                  int N, int N2, int S, const float* l0, int l0_row, const float* feat, float* m0,
                                  long long* labels0, float* inj, int B, int K, int F, void* stream);

/* ---- the mean-field logit noise drawn on the device (MeanFieldDistribution.sample, cub/code/nn.py:1421-1427) ----
 * The training step samples its logits as l = mean + noise_level * N(0,1) (model.py:420-421).  The N(0,1) draw here is a
 * pure function of (seed, draw, global pixel, part), defined in csrc/canon_math.cuh: Philox4x32-10 with key = seed and
 * counter = (global pixel lo, hi, part / 4, draw), 24-bit uniforms in (0, 1], Box-Muller with the canonical log / sin /
 * cos.  It does not depend on K, the launch geometry or the batch split.  draw = 0 for l0, 1 for l1; global pixel =
 * (sample_offset + b) * P + p.  The sampled logit is fl(mean + fl(noise_level * z)); -inf (a padded part) stays -inf. */
/* eps [n_pix, K] for global pixels pix_offset .. pix_offset + n_pix - 1: what the kernels below draw. */
int ups_normal_philox_fwd(unsigned long long seed, int draw, long long pix_offset, long long n_pix, int K, float* out,
                          void* stream);
/* ups_part_softmax_sampled_fwd with eps drawn in registers (pixel i of `mean` is global pixel pix_offset + i);
 * logits_out, labels and hard may be NULL. */
int ups_part_softmax_sampled_philox_fwd(const float* mean, unsigned long long seed, int draw, long long pix_offset,
                                        float noise_level, float* logits_out, float* probs, int64_t* labels, float* hard,
                                        long long n_pix, int K, void* stream);
/* The fused forward kernels on means: the arguments of the _rows forms, then (seed, sample_offset, noise_level).  l0 / l1
 * are the means; the noise is added right after the load (decode side draw 0, encode side draw 1).  The sampled logits
 * are not written: ups_normal_philox_fwd + ups_mean_field_sample_fwd regenerate them bit for bit.  The backward entry
 * points are unchanged: d l / d mean is the identity, so dl0 / dl1 are the gradients of the means. */
int ups_step_decode_fwd_noise(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0, float* inj,
                              int B, int P, int K, int F, unsigned long long seed, long long sample_offset, float noise_level,
                              void* stream);
int ups_step_encode_fwd_noise(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm, float* pooled,
                              int B, int P, int K, int Kpl, void* ws, size_t ws_bytes, unsigned long long seed,
                              long long sample_offset, float noise_level, void* stream);
int ups_step_warp_decode_fwd_noise(const float* U, const float* U2, const float* coord, const float* T, float* out,
                                   float* out2, int N, int N2, int S, const float* l0, int l0_row, const float* feat, float* m0,
                                   long long* labels0, float* inj, int B, int K, int F, unsigned long long seed,
                                   long long sample_offset, float noise_level, void* stream);
/* The same draws with the seed read from device memory: `seed` points to one device word (the uint64 seed, e.g. a
 * one-element int64 tensor holding the same bits) that the kernel loads once, in its prologue.  For equal seed values the
 * results are bit-identical to the by-value forms above.  A launch captured in a CUDA graph keeps the pointer, not the
 * value: writing a new seed into the word before a replay gives that replay a new draw. */
int ups_normal_philox_fwd_dseed(const unsigned long long* seed, int draw, long long pix_offset, long long n_pix, int K,
                                float* out, void* stream);
int ups_part_softmax_sampled_philox_fwd_dseed(const float* mean, const unsigned long long* seed, int draw,
                                              long long pix_offset, float noise_level, float* logits_out, float* probs,
                                              int64_t* labels, float* hard, long long n_pix, int K, void* stream);
int ups_step_decode_fwd_noise_dseed(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0,
                                    float* inj, int B, int P, int K, int F, const unsigned long long* seed,
                                    long long sample_offset, float noise_level, void* stream);
int ups_step_encode_fwd_noise_dseed(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm,
                                    float* pooled, int B, int P, int K, int Kpl, void* ws, size_t ws_bytes,
                                    const unsigned long long* seed, long long sample_offset, float noise_level, void* stream);

/* K1 + K3 of the fused step in ONE launch (csrc/step_fwd_fused.cu): the TPS warp of the views (ups_tps_warp_pair_fwd's
 * arguments: U [N,S,S,3], optional second image set U2 [N2,S,S,3] sharing the first N2 warps, coord, T -> out, out2) and
 * the decode-side forward (ups_step_decode_fwd's arguments) are independent (model.py:282-311 vs :426-447,482-484);
 * their CTAs are interleaved in one grid so that the warp's arithmetic hides under the decode side's memory stream.
 * Results are bit-identical to the two separate calls.  K in {8,16,32}, F in {16,32,64}, S*S % 32 == 0. */
int ups_step_warp_decode_fwd(const float* U, const float* U2, const float* coord, const float* T, float* out, float* out2,
                             int N, int N2, int S, const float* l0, const float* feat, float* m0, long long* labels0,
                             float* inj, int B, int K, int F, void* stream);

/* ---- data-parallel step wrapper (SURVEY.md 8d "DP step", 8e) ------------------------------------------------
 * The reference trains on one GPU; the only multi-GPU analogue in its tree is the IMM baseline's host-side tower
 * averaging (baselines/imm/imm/train/cnn_train_multi.py:75-118, `average_gradients`).  ups_dp_allreduce is that mean
 * over ranks as ONE kernel over NVLink peer memory, in place on a bucket of the flat gradient buffer:
 *   peer_bufs    HOST array [world] of this process's device mappings of every rank's bucket (entry `rank` = own)
 *   mc_buf       device mapping of the multicast object bound to all buckets (NVSwitch in-switch reduction), or NULL:
 *                then the kernel reads and writes the peers' buckets through peer_bufs
 *   peer_signals HOST array [world] of mappings of every rank's signal pad: ups_dp_allreduce_signal_bytes(world, n_ctas)
 *                bytes, zero-initialised once by its owner before the first call (the barriers reset it themselves)
 *   scale        applied to the sum (1/world for the mean); n_floats % 4 == 0; n_ctas CTAs of 128 threads, <= 42 registers,
 *                no shared memory (sized to co-reside with the persistent K4 grid)
 * All ranks must enqueue the call with the same n_floats/n_ctas; the kernel waits (device side, no host sync) until
 * every rank's call has started, i.e. until the producers of every rank's bucket have finished in stream order. */
int ups_dp_allreduce(void* const* peer_bufs, void* mc_buf, void* const* peer_signals, int rank, int world,
                     long long n_floats, float scale, int n_ctas, void* stream);
size_t ups_dp_allreduce_signal_bytes(int world, int n_ctas);

/* Stand-in parameterised modules that produce the gradients the wrapper all-reduces (csrc/standin.cu).
 * encoder tail: feat[b,k,:] = pooled[b,k,:] . Wlin[C,F] + blin[F]         cub/code/SB_model48i/model.py:50-52
 *   bwd: out = [dWlin (C*F), dblin (F)] from pooled [B,K,C] (C == 3) and dfeat [B,K,F]
 * decoder head: recon[b,p,:] = concat(feat[b,label,:], one_hot(label)) . Whead[F+K,3] + bhead[3]
 *   (1x1 conv on nn.unpool_features_gathered's injection, cub/code/nn.py:2469-2487; labels int64 [B,P])
 *   bwd: out = [dWhead ((F+K)*3), dbhead (3)] from g_recon [B,P,3], labels, feat [B,K,F]
 * Fixed-order sums (deterministic).  ws from ups_standin_workspace_bytes. */
int ups_standin_tail_fwd(const float* pooled, const float* Wlin, const float* blin, float* feat, int B, int K, int C,
                         int F, void* stream);
int ups_standin_tail_bwd(const float* pooled, const float* dfeat, float* dWlin_dblin, int B, int K, int C, int F,
                         void* ws, size_t ws_bytes, void* stream);
int ups_standin_head_fwd(const long long* labels, const float* feat, const float* Whead, const float* bhead,
                         float* recon, int B, int P, int K, int F, void* stream);
int ups_standin_head_bwd(const float* g_recon, const long long* labels, const float* feat, float* dWhead_dbhead, int B,
                         int P, int K, int F, void* ws, size_t ws_bytes, void* stream);
size_t ups_standin_workspace_bytes(int B, int P, int K, int F);

#ifdef __cplusplus
}
#endif
#endif /* UPS_B200_H */
