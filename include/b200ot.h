/* b200ot.h — C ABI of the B200-native Sinkhorn / kernel-MMD reduction engine.
 *
 * This is the drop-in boundary for the hot path of jeanfeydy/geomloss (reference commit 00e493f).
 * The reference has no FFI: its plugin seams are the Python callables
 *   softmin(eps, C_xy, h_y) -> f_x            (src/geomloss/_legacy/sinkhorn_divergence.py:291-303,
 *                                              implemented by softmin_tensorized / softmin_online,
 *                                              src/geomloss/_legacy/sinkhorn_samples.py:32-71,337-346)
 *   kernel matvecs of kernel_loss             (src/geomloss/_legacy/kernel_samples.py:92-146)
 * which the pykeops "online" backend lowers to one CUDA map-reduce launch per call
 * (sinkhorn_samples.py:322-334: generic_logsumexp("(B - (P * cost))", Vi(1), Vi(D), Vj(D), Vj(1), Pm(1))).
 * The functions below are what a maintainer would bind in place of that pykeops call.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to fp32 (or the stated type), row-major, contiguous;
 *     the caller owns every buffer; nothing is allocated, freed or retained by the library;
 *   - kernels are enqueued on `stream` (a cudaStream_t passed as void*) and the call returns
 *     immediately; no host synchronisation happens inside;
 *   - return value: 0 on success, a negative B200OT_E* code otherwise (never throws, never aborts);
 *   - "rows" x:(N,D) own the output, "cols" y:(M,D) are reduced over; D <= B200OT_MAX_D;
 *   - a reduction is split into two launches so that the column cloud can be packed once and
 *     reused (and so that partial results of column shards living on other GPUs can be merged):
 *         pack  ->  partial reduction  ->  finalize.
 *
 * Environment variables (read by the one-call entry points on every call; meant for A/B timing and for the parity tests
 * that hold both settings of every switch to the oracle — a deployment leaves them unset):
 *   B200OT_TC_MIN_D      "d" or "softmin_fwd,softmin_bwd,conv_fwd,conv_bwd": smallest D <= B200OT_MAX_D an operator
 *                        hands to the tensor-core kernels (default "6,9,5,9": forward softmin from 6, gaussian from 5)
 *   B200OT_TC_MIN_PAIRS  smallest N*M for that hand-over (default 8e8)
 *   B200OT_TC_BWD        "p_terms,epilogue_warps,ldall,merge" of the tensor-core row-gradient kernel (default "2,8,0,1")
 */
#ifndef B200OT_H_
#define B200OT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B200OT_API __attribute__((visibility("default")))
#else
#define B200OT_API
#endif

#define B200OT_VERSION 202 /* 0.2.2 */
#define B200OT_MAX_D 8     /* dimensions served by the CUDA-core (register tile) kernels of this build */

/* error codes */
#define B200OT_OK 0
#define B200OT_EINVAL -1   /* bad argument (null pointer, non-positive size, unsupported p / D / kind) */
#define B200OT_ESCRATCH -2 /* scratch buffer too small (see *_scratch_bytes) */
#define B200OT_ECUDA -3    /* a CUDA runtime call failed; see b200ot_last_cuda_error() */
#define B200OT_EALIGN -4   /* pointer not 16-byte aligned */

/* kernel kinds for b200ot_kernel_conv_* (reference: kernel_samples.py:62-82) */
#define B200OT_KERNEL_GAUSSIAN 0  /* exp(-|x-y|^2 / (2 blur^2)) */
#define B200OT_KERNEL_LAPLACIAN 1 /* exp(-sqrt(max(|x-y|^2/blur^2, 1e-8))) */
#define B200OT_KERNEL_ENERGY 2    /* -sqrt(max(|x-y|^2, 1e-8)) */

/* The reference has TWO conventions for the Euclidean norm under p = 1 / laplacian / energy:
 *   backend="tensorized":  sqrt(clamp_min(|x-y|^2, 1e-8))   (utils.py:56-61)           -> p = 1, kinds 1, 2
 *   backend="online" / "multiscale" (pykeops Norm2 / .sqrt(), sinkhorn_samples.py:303-306, utils.py:56-58):
 *                          sqrt(|x-y|^2), zero gradient at coincident points            -> flag below
 * Or the flag into `p` (softmin entry points) or `kind` (kernel_conv entry points). */
#define B200OT_P_UNCLAMPED 0x100
#define B200OT_KERNEL_UNCLAMPED 0x100

B200OT_API const char* b200ot_strerror(int code);
B200OT_API const char* b200ot_last_cuda_error(void);
B200OT_API int b200ot_version(void);

/* ---------------------------------------------------------------------------------------------
 * Softmin  —  out_i = -eps * log sum_j exp( h_j - |x_i - y_j|^p / (p * eps) ),   p in {1, 2}
 * replaces softmin_tensorized (sinkhorn_samples.py:32-71) / softmin_online (:337-346).
 * p = 1 uses sqrt(max(|x-y|^2, 1e-8)) like the reference's `distances` (utils.py:56-61);
 * p = 1 | B200OT_P_UNCLAMPED uses the pykeops convention (see above).
 * ------------------------------------------------------------------------------------------- */

/* Bytes of scratch needed by b200ot_softmin_fwd / _bwd_x for (N rows, M cols, D). */
B200OT_API int64_t b200ot_softmin_scratch_bytes(int64_t N, int64_t M, int32_t D);

/* One-call softmin:  out (N) <- alpha_old * out_old + beta * softmin(eps, (x, y), h)
 *   h_a (M), h_b (M, nullable):  h_j = h_a[j] + h_scale_b * h_b[j]
 *       (the Sinkhorn loop's  b_log + g / eps  is h_a = b_log, h_b = g, h_scale_b = 1/eps —
 *        sinkhorn_divergence.py:480-488 — fused here instead of a separate elementwise launch);
 *   out_old (N, nullable), alpha_old, beta:  the damping and the 1/2 (f + ft) averaging of
 *       sinkhorn_divergence.py:480-493 fused into the epilogue (alpha_old=0, beta=1: plain softmin);
 *   lse2_out (N, nullable): log2-domain log-sum-exp per row, saved for the backward pass;
 *   center (D, nullable): device vector subtracted from both clouds before the |x|^2 - 2x.y + |y|^2
 *       expansion (improves fp32 conditioning; any point near the data works, zeros if null);
 *   scratch: >= b200ot_softmin_scratch_bytes(N, M, D) bytes, 16-byte aligned.
 */
B200OT_API int b200ot_softmin_fwd(const float* x, const float* y, const float* h_a, const float* h_b, float h_scale_b,
                       const float* center, const float* out_old, float alpha_old, float beta, float* out,
                       float* lse2_out, int64_t N, int64_t M, int32_t D, int32_t p, float eps, void* scratch,
                       int64_t scratch_bytes, void* stream);

/* Gradient of the softmin w.r.t. the row cloud (the only gradient the reference's autograd
 * contract carries: columns and h are detached, sinkhorn_samples.py:179-185, sinkhorn_divergence.py:616-623):
 *   grad_x[i,:] = grad_out[i] * sum_j softmax_j(h_j - C_ij/eps) * dC(x_i, y_j)/dx_i
 * lse2 is the lse2_out of the matching forward call.  grad_x (N,D) is overwritten. */
B200OT_API int b200ot_softmin_bwd_x(const float* x, const float* y, const float* h_a, const float* h_b, float h_scale_b,
                         const float* center, const float* lse2, const float* grad_out, float* grad_x, int64_t N,
                         int64_t M, int32_t D, int32_t p, float eps, void* scratch, int64_t scratch_bytes,
                         void* stream);

/* --- the three stages of b200ot_softmin_fwd, exposed for column-sharded (multi-GPU) use --- */

/* Number of floats of a packed column buffer for M columns of dimension D with `extra` per-column
 * scalars (softmin: 1 = h; gaussian conv: 2 = -|y|^2/2 and weight; laplacian / energy conv: 1 = weight). */
B200OT_API int64_t b200ot_packed_cols_floats(int64_t M, int32_t D, int32_t extra);

/* Pack the column cloud for a softmin at temperature eps (coordinates pre-scaled, h folded into the
 * per-column term, padding columns neutral).  cols_out: b200ot_packed_cols_floats(M, D, 1) floats. */
B200OT_API int b200ot_softmin_pack(const float* y, const float* h_a, const float* h_b, float h_scale_b, const float* center,
                        int64_t M, int32_t D, int32_t p, float eps, float* cols_out, void* stream);

/* Number of column splits the partial reduction will use for (N, M, D): partials hold n_split * N pairs. */
B200OT_API int32_t b200ot_softmin_num_splits(int64_t N, int64_t M, int32_t D);

/* Partial reduction over the packed columns: part[(s*N + i)*2 + {0,1}] = (running max m, sum of
 * exp2(t - m)) in the log2 domain, for s < n_split.  This is the kernel that does the N x M work. */
B200OT_API int b200ot_softmin_partial(const float* x, const float* center, const float* cols, float* part, int32_t n_split,
                           int64_t N, int64_t M, int32_t D, int32_t p, float eps, void* stream);

/* ---- ranges mode: block-sparse and batched problems in ONE launch ------------------------------------------
 * Replaces the reference's `ranges=` argument of pykeops reductions (softmin_multiscale, sinkhorn_samples.py:445-450,
 * built by kernel_truncation :493-530 / from_matrix; kernel_multiscale, kernel_samples.py:246-256) and the batched
 * LazyTensor reduction of softmin_online_lazytensor (:229-290, a block-diagonal problem).
 *   segment  = a run of consecutive rows that share one list of column pieces (one CTA per segment):
 *              a cluster of the sorted row cloud (cut into <= max_rows_per_segment rows), or a batch element;
 *   piece    = a run of consecutive column SLOTS (col_start, col_count), both multiples of col_align,
 *              col_count <= max_cols_per_piece;
 *   slots    = the packed column buffer in gather mode: slot s holds column src_index[s] of the caller's arrays,
 *              or a neutral padding column when src_index[s] < 0 — clusters / batch elements are padded to a
 *              multiple of col_align slots so that every piece starts on a chunk boundary.
 * The reduction visits exactly the (row, column) pairs listed: bit-for-bit the blocks of the reference's ranges. */
typedef struct { int32_t row_start, row_count, piece_begin, piece_end; } b200ot_segment; /* 16-byte aligned array */
typedef struct { int32_t col_start, col_count; } b200ot_piece;                           /*  8-byte aligned array */
#define B200OT_RANGES_BIG 0   /* 512-row segments, pieces <= 1024 columns: large clusters */
#define B200OT_RANGES_SMALL 1 /* 128-row segments, pieces <= 256 columns: small clusters / small batch elements */
B200OT_API void b200ot_ranges_shape(int32_t variant, int32_t* max_rows_per_segment, int32_t* max_cols_per_piece,
                                    int32_t* col_align);

/* b200ot_softmin_pack in gather mode: cols_out holds b200ot_packed_cols_floats(n_slots, D, 1) floats. */
B200OT_API int b200ot_softmin_pack_gather(const float* y, const float* h_a, const float* h_b, float h_scale_b,
                                          const float* center, const int32_t* src_index, int64_t n_slots, int32_t D,
                                          int32_t p, float eps, float* cols_out, void* stream);

/* part: (N, 2) (m, s) pairs, one per row; rows that belong to no segment are left untouched. */
B200OT_API int b200ot_softmin_partial_ranges(const float* x, const float* center, const float* cols,
                                             const b200ot_segment* seg, int64_t n_seg, const b200ot_piece* pieces,
                                             float* part, int64_t N, int32_t D, int32_t p, float eps,
                                             int32_t variant, void* stream);

/* Collapse n_part partial (m, s) sets into one per row: merged[i*2 + {0,1}].  A rank calls this on its own
 * splits before exchanging partials with the other column shards (N*8 bytes per rank). */
B200OT_API int b200ot_softmin_merge(const float* part, int32_t n_part, float* merged, int64_t N, void* stream);

/* Merge n_part partial (m, s) sets (own splits and/or other ranks' shards, concatenated along the
 * leading axis) and apply the epilogue of b200ot_softmin_fwd. */
B200OT_API int b200ot_softmin_finalize(const float* part, int32_t n_part, const float* out_old, float alpha_old, float beta,
                            float* out, float* lse2_out, int64_t N, float eps, void* stream);

/* --- stages of b200ot_softmin_bwd_x, for column-sharded use: per-shard partial sums
 *     part[(s*N + i)*(D+1) + {0: sum_j w_ij, 1+k: sum_j w_ij * (coordinate or unit-vector term)}],
 *     which add across shards (all-reduce SUM) before the finalize --- */
B200OT_API int b200ot_softmin_bwd_partial(const float* x, const float* center, const float* cols, const float* lse2,
                                          float* part, int32_t n_split, int64_t N, int64_t M, int32_t D, int32_t p,
                                          float eps, void* stream);
/* ranges variant (see b200ot_softmin_partial_ranges): part is (N, D+1), one split */
B200OT_API int b200ot_softmin_bwd_partial_ranges(const float* x, const float* center, const float* cols,
                                                 const float* lse2, const b200ot_segment* seg, int64_t n_seg,
                                                 const b200ot_piece* pieces, float* part, int64_t N, int32_t D,
                                                 int32_t p, float eps, int32_t variant, void* stream);
/* One call: sums (N, D+1) = the merged partial sums of the row-gradient pass over ALL columns given (pack + partial +
 * merge; CUDA-core path for D <= B200OT_MAX_D, tensor-core path for p = 2 up to D = 64).  A column shard calls this
 * on its slice, all-reduces `sums` (SUM) and finishes with b200ot_softmin_bwd_finalize(n_part = 1). */
B200OT_API int b200ot_softmin_bwd_sums(const float* x, const float* y, const float* h_a, const float* h_b,
                                       float h_scale_b, const float* center, const float* lse2, float* sums,
                                       int64_t N, int64_t M, int32_t D, int32_t p, float eps, void* scratch,
                                       int64_t scratch_bytes, void* stream);
/* merged[i*width + a] = sum_s part[(s*N + i)*width + a] */
B200OT_API int b200ot_rowsum_merge(const float* part, int32_t n_part, int32_t width, float* merged, int64_t N,
                                   void* stream);
B200OT_API int b200ot_softmin_bwd_finalize(const float* part, int32_t n_part, const float* x, const float* center,
                                           const float* grad_out, float* grad_x, int64_t N, int32_t D, int32_t p,
                                           float eps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Kernel convolution  —  out_i = sum_j k(x_i, y_j) * w_j      (kernel_samples.py:128-137)
 * ------------------------------------------------------------------------------------------- */
/* Forward and row gradients additionally accept 8 < D <= 64 for every kind: that range runs on the tensor cores
 * (tcgen05, fp16x2 split operands, -|x - y|^2 / 2 accumulated in TMEM; laplacian / energy take the square root in the
 * epilogue, on coordinates scaled by the extent of the clouds, with or without B200OT_KERNEL_UNCLAMPED).  For
 * D <= B200OT_MAX_D the library picks the faster of the two paths per operator and problem size for the gaussian
 * (csrc/b200ot_kernel_conv.cu: tc_routed); laplacian / energy stay on the CUDA cores there.  Results agree to the
 * tolerances of DESIGN.md section 4 either way. */
B200OT_API int64_t b200ot_kernel_conv_scratch_bytes(int64_t N, int64_t M, int32_t D);

B200OT_API int b200ot_kernel_conv_fwd(const float* x, const float* y, const float* w, const float* center, float* out,
                           int64_t N, int64_t M, int32_t D, int32_t kind, float blur, void* scratch,
                           int64_t scratch_bytes, void* stream);

/* grad_x[i,:] = grad_out[i] * sum_j w_j * d k(x_i, y_j) / d x_i   (rows only; columns via a swapped call) */
B200OT_API int b200ot_kernel_conv_bwd_x(const float* x, const float* y, const float* w, const float* center,
                             const float* grad_out, float* grad_x, int64_t N, int64_t M, int32_t D, int32_t kind,
                             float blur, void* scratch, int64_t scratch_bytes, void* stream);

/* Value AND unit row gradient from ONE pass over the N x M pairs (gaussian only; EINVAL otherwise):
 *   out[i] = sum_j k(x_i, y_j) w_j,    grad_unit[i,:] = sum_j w_j * d k(x_i, y_j) / d x_i
 * i.e. b200ot_kernel_conv_fwd and b200ot_kernel_conv_bwd_x(grad_out = 1) together: the row-gradient reduction
 * accumulates sum_j w_j k_ij anyway, so a caller that will differentiate (autograd of kernel_loss's matvecs,
 * kernel_samples.py:116-137) saves the separate forward reduction and multiplies grad_unit by its upstream gradient
 * row by row.  Same scratch size as the other two. */
B200OT_API int b200ot_kernel_conv_fwd_bwd_x(const float* x, const float* y, const float* w, const float* center,
                                 float* out, float* grad_unit, int64_t N, int64_t M, int32_t D, int32_t kind,
                                 float blur, void* scratch, int64_t scratch_bytes, void* stream);

/* --- stages of the CUDA-core kernel convolutions (D <= B200OT_MAX_D), ranges mode: truncated block-sparse
 *     MMDs (kernel_multiscale, kernel_samples.py:177-271) and batched problems.  cols: gather-packed,
 *     b200ot_packed_cols_floats(n_slots, D, 2) floats.  part: (N) sums (backward = 0) or (N, width) sums
 *     (backward = 1; width = D + 1 for the gaussian kernel, D otherwise); partial sums of column shards add. --- */
B200OT_API int b200ot_kernel_conv_pack_gather(const float* y, const float* w, const float* center,
                                              const int32_t* src_index, int64_t n_slots, int32_t D, int32_t kind,
                                              float blur, float* cols_out, void* stream);
B200OT_API int b200ot_kernel_conv_partial_ranges(const float* x, const float* center, const float* cols,
                                                 const b200ot_segment* seg, int64_t n_seg,
                                                 const b200ot_piece* pieces, float* part, int64_t N, int32_t D,
                                                 int32_t kind, float blur, int32_t backward, int32_t variant,
                                                 void* stream);
/* out_i = sign(kind) * sum_s part[s*N + i] */
B200OT_API int b200ot_kernel_conv_finalize(const float* part, int32_t n_part, float* out, int64_t N, int32_t kind,
                                           void* stream);
/* grad_x from n_part sets of (N, width) row-gradient sums */
B200OT_API int b200ot_kernel_conv_bwd_finalize(const float* part, int32_t n_part, const float* x, const float* center,
                                               const float* grad_out, float* grad_x, int64_t N, int32_t D,
                                               int32_t kind, float blur, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Small problems: one launch per symmetric Sinkhorn iteration
 * replaces the four softmin calls of the loop body of sinkhorn_loop (sinkhorn_divergence.py:468-493) — and of its
 * initialisation (:461-465) and final gradient-carrying step (:612-623) — for B stacked problems
 * x:(B,N,D) y:(B,M,D) a_log:(B,N) b_log:(B,M) with N, M <= B200OT_SMALL_MAX_POINTS, D <= B200OT_MAX_D:
 *     f_ba_out <- alpha_old f_ba + beta softmin(eps, (x, y), b_log + g_ab/eps)      (B,N)
 *     g_ab_out <- alpha_old g_ab + beta softmin(eps, (y, x), a_log + f_ba/eps)      (B,M)
 *     f_aa_out <- alpha_old f_aa + beta softmin(eps, (x, x), a_log + f_aa/eps)      (B,N)   (debiasing; nullable pair)
 *     g_bb_out <- alpha_old g_bb + beta softmin(eps, (y, y), b_log + g_bb/eps)      (B,M)
 * all four reading the OLD potentials (f_ba .. g_bb all null: h = log-weights, the initialisation; alpha_old = 0).
 * a_log / b_log are natural-log weights, or the weights themselves when weights_linear = 1.
 * Outputs must not alias inputs.  lse2_out (nullable): B*(2N+2M) floats [f_ba | g_ab | f_aa | g_bb], the log2-domain
 * log-sum-exp of every row, consumed by b200ot_sinkhorn_final_bwd_small:
 *     grad_x <- scale_out * ( go_f_ba[i] d softmin_xy / d x_i + go_f_aa[i] d softmin_xx / d x_i )     (B,N,D)
 *     grad_y <- scale_out * ( go_g_ab[j] d softmin_yx / d y_j + go_g_bb[j] d softmin_yy / d y_j )     (B,M,D)
 * with columns and potentials held constant (the reference's autograd contract); f_ba .. g_bb are the potentials
 * that entered the final step; go_* nullable (zero upstream gradient).
 * ------------------------------------------------------------------------------------------- */
#define B200OT_SMALL_MAX_POINTS 65536
B200OT_API int b200ot_sinkhorn_iteration_small(const float* x, const float* y, const float* a_log, const float* b_log,
                                               const float* f_ba, const float* g_ab, const float* f_aa,
                                               const float* g_bb, float* f_ba_out, float* g_ab_out, float* f_aa_out,
                                               float* g_bb_out, float* lse2_out, int64_t B, int64_t N, int64_t M,
                                               int32_t D, int32_t p, float eps, float alpha_old, float beta,
                                               int32_t weights_linear, void* stream);
/* The whole descent in ONE host call: initialisation at eps_list[0] (potentials <- damped softmins of the log-weights)
 * followed by one averaged symmetric update per temperature of eps_list (host array of n_eps doubles) — n_eps + 1
 * launches enqueued back to back, no Python / FFI round trip between them.  rho <= 0: balanced (damping 1), else
 * damping 1/(1 + eps/rho) per temperature (sinkhorn_divergence.py:56-58).  pots_a, pots_b: two scratch sets of
 * B*(2N+2M) floats [f_ba | g_ab | f_aa | g_bb] used as ping-pong buffers; *result_in_a tells which one holds the final
 * iterate.  weights_linear = 1: a, b are the weights themselves (log taken in the kernel, -100000 floor for a <= 0). */
B200OT_API int b200ot_sinkhorn_loop_small(const float* x, const float* y, const float* a, const float* b,
                                          int32_t weights_linear, const double* eps_list, int32_t n_eps, double rho,
                                          int32_t debias, float* pots_a, float* pots_b, int32_t* result_in_a,
                                          int64_t B, int64_t N, int64_t M, int32_t D, int32_t p, void* stream);
B200OT_API int b200ot_sinkhorn_final_bwd_small(const float* x, const float* y, const float* a_log, const float* b_log,
                                               const float* f_ba, const float* g_ab, const float* f_aa,
                                               const float* g_bb, const float* lse2, const float* go_f_ba,
                                               const float* go_g_ab, const float* go_f_aa, const float* go_g_bb,
                                               float* grad_x, float* grad_y, int64_t B, int64_t N, int64_t M,
                                               int32_t D, int32_t p, float eps, float scale_out,
                                               const float* go_scale, int32_t weights_linear, void* stream);
/* go_scale (nullable): (B,) per-problem factor applied to every go_* — the upstream gradient of the B loss values when
 * go_* hold d value / d potential as written by b200ot_sinkhorn_cost_small.
 *
 * sinkhorn_cost (sinkhorn_divergence.py:165-255) of B stacked small problems in one launch, one value per problem:
 *     rho <= 0 (balanced):  value = <a, f_ba - f_aa> + <b, g_ab - g_bb>
 *     rho  > 0:             value = <a, w (e^{-f_aa/rho} - e^{-f_ba/rho})> + <b, w (e^{-g_bb/rho} - e^{-g_ab/rho})>,
 *                           w = rho + eps/2
 * (f_aa = g_bb = NULL: no debiasing — <a, f_ba> + <b, g_ab>, resp. w (1 - e^{-f/rho}).)  Nullable outputs: go_* =
 * d value / d potential per point, phi (B,N) / psi (B,M) = d value / d a_i, d value / d b_j. */
B200OT_API int b200ot_sinkhorn_cost_small(const float* a, const float* b, const float* f_ba, const float* g_ab,
                                          const float* f_aa, const float* g_bb, int64_t B, int64_t N, int64_t M,
                                          float rho, float eps, float* value, float* go_f_ba, float* go_g_ab,
                                          float* go_f_aa, float* go_g_bb, float* phi, float* psi, void* stream);

/* value[b] = 1/2 <a, a_x> + 1/2 <b, b_y> - <a, b_x> (kernel_samples.py:139-146) from the outputs of
 * b200ot_kernel_mmd_small, one launch, fixed summation order. */
B200OT_API int b200ot_kernel_mmd_value_small(const float* a, const float* b, const float* a_x, const float* b_y,
                                             const float* b_x, int64_t B, int64_t N, int64_t M, float* value,
                                             void* stream);

/* Bounding box of the rows of x:(n,D) and y:(m,D) (m = 0: x alone), D <= B200OT_MAX_D: lo_hi[0..D) = minima,
 * lo_hi[D..2D) = maxima — the inputs of max_diameter (sinkhorn_divergence.py:96-112) in one launch.  scratch:
 * b200ot_cloud_extent_scratch_bytes() bytes, ZERO before its first use (the kernel leaves it reusable). */
B200OT_API int64_t b200ot_cloud_extent_scratch_bytes(void);
B200OT_API int b200ot_cloud_extent(const float* x, int64_t n, const float* y, int64_t m, int32_t D, float* lo_hi,
                                   void* scratch, int64_t scratch_bytes, void* stream);

/* Kernel norms on small clouds (same size limits): the matvecs of kernel_loss (kernel_samples.py:116-137) in one launch,
 *     a_x = K(x,x) a   b_y = K(y,y) b   b_x = K(x,y) b   a_y = K(y,x) a  (a_y nullable: only needed for potentials / d/db)
 * and the gradient of  value = 1/2 <a, a_x> + 1/2 <b, b_y> - <a, b_x>  w.r.t. both clouds, with the reference's
 * DoubleGrad / detach pattern (kernel_samples.py:43-54, :116-146), scaled by grad_value[batch], in one more. */
B200OT_API int b200ot_kernel_mmd_small(const float* x, const float* y, const float* a, const float* b, float* a_x,
                                       float* b_y, float* b_x, float* a_y, int64_t B, int64_t N, int64_t M, int32_t D,
                                       int32_t kind, float blur, void* stream);
B200OT_API int b200ot_kernel_mmd_bwd_small(const float* x, const float* y, const float* a, const float* b,
                                           const float* grad_value, float* grad_x, float* grad_y, int64_t B, int64_t N,
                                           int64_t M, int32_t D, int32_t kind, float blur, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Grid softmin  —  the separable soft-C-transform on (batch, N, N[, N]) images / volumes
 * replaces softmin_grid (src/geomloss/_legacy/utils.py:190-279), the operator of the image Sinkhorn loop
 * (src/geomloss/_legacy/sinkhorn_images.py:26-202):
 *   out <- alpha_old * out_old + beta * ( -eps * LSE over the whole grid of  h - |x - y|^p / (p eps) ),
 *   h = h_a + h_scale_b * h_b (h_b nullable), pixel coordinates arange(N)/N, p in {1, 2}, dim in {1, 2, 3}.
 * `out` must not alias an input (the per-axis passes run in place on it).  N <= 1024.
 * ------------------------------------------------------------------------------------------- */
B200OT_API int b200ot_softmin_grid(const float* h_a, const float* h_b, float h_scale_b, const float* out_old,
                                   float alpha_old, float beta, float* out, int64_t batch, int32_t N, int32_t dim,
                                   int32_t p, float eps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pipe-ceiling micro-benchmarks (used by bench.py to measure the MUFU / FP32 roofline of the
 * device it runs on; each launches one kernel doing `iters` dependent steps per thread and
 * returns the number of operations executed per thread-step through *ops_per_thread_iter).
 * ------------------------------------------------------------------------------------------- */
#define B200OT_UBENCH_MUFU_EX2 0
#define B200OT_UBENCH_FFMA 1
#define B200OT_UBENCH_FFMA2 2
B200OT_API int b200ot_ubench(int32_t which, int32_t iters, int32_t blocks, float* sink, int32_t* ops_per_thread_iter,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200OT_H_ */
