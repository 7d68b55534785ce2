/*
 * gfs3d.h -- C ABI of the B200-native (sm_100a) hot path of GFS-3DSeg_GWs.
 *
 * The reference (Pixie8888/GFS-3DSeg_GWs) is pure PyTorch and has no FFI of its own; its boundary for this path
 * is the Python module API of model/dgcnn.py and model/capl.py plus the sklearn KMeans call in get_basis.py.
 * Each entry point below names the reference lines whose arithmetic it replaces.  The Python drop-in modules in
 * gfs-3dseg_gws_b200/model/ call these through ctypes (gfs-3dseg_gws_b200/gfs3d/_lib.py); INTEGRATION.md shows the
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless its name ends in _host
 *   - the caller owns all memory (outputs and workspaces are caller-allocated); the library never allocates,
 *     frees or retains device memory
 *   - every call enqueues asynchronously on `stream` (a cudaStream_t passed as void*) and never synchronises
 *   - every call returns 0 on success, or a gfs_status code; gfs_last_error_string() describes the last failure
 *     of the calling thread.  There is no CPU fallback anywhere.
 *   - "cm"  = channel-major fp32 activations  (B, C, N) with an explicit batch stride in elements
 *   - "act" = bf16 activation matrix in the tiled layout described below
 *
 * bf16 "act" layout (memory laid out for tcgen05: a tile is bulk-copied by TMA straight into a UMMA operand)
 *   logical matrix (M rows = points b*N+n, Kc columns), M padded to 128, Kc a multiple of 64;
 *   stored as tiles [M/128][Kc/64], each tile 128 rows x 64 bf16 = 16 KiB in the canonical K-major SWIZZLE_128B
 *   arrangement:  byte(r, c) = r*128 + (((c/8) ^ (r&7)) << 4) + (c%8)*2.
 *   weights use the same arrangement with [Kc/64] tiles of R rows x 64 bf16 (see gfs_pack_weight_bf16).
 */
#ifndef GFS3D_H
#define GFS3D_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    GFS_OK = 0,
    GFS_ERR_BAD_ARG = 1,       /* null pointer / non-positive size / misaligned pointer */
    GFS_ERR_UNSUPPORTED = 2,   /* a width / size this build does not specialise (raised, never silently emulated) */
    GFS_ERR_CUDA = 3           /* a CUDA runtime error; the string carries cudaGetErrorString */
} gfs_status;

enum { GFS_ACT_NONE = 0, GFS_ACT_LRELU02 = 1, GFS_ACT_RELU = 2 };

int gfs_version(void);
const char* gfs_last_error_string(void);
/* number of SMs of the current device (grid sizing of the persistent kernels); <0 on error */
int gfs_device_sm_count(void);
/* Programmatic dependent launch of the inference kernels (on by default; GFS3D_PDL=0 in the environment or
 * gfs_set_pdl(0) turn it off): each kernel of a call chain may become resident while its predecessor on the stream
 * drains and blocks in its first statement (griddepcontrol.wait) until the predecessor has completed, so the launch
 * latency of ~45 kernels per forward pass (model/capl.py:170-192) overlaps the previous kernel's tail.  Stream
 * semantics and results are unchanged; capturable into CUDA graphs.                                                */
int gfs_set_pdl(int on);

/* ---- kNN graph: model/dgcnn.py:17-23 (knn) -------------------------------------------------------------------
 * d(i,j) = -|x_i|^2 + 2 x_i.x_j - |x_j|^2 in fp32 with the pinned order of oracle/gfs_oracle.c; the k largest per
 * row, nearest first, ties -> ascending index.  The N x N matrix is never written to memory.
 *   x        cm fp32, channel stride N, batch stride x_bstride (elements); C <= 64, N % 4 == 0
 *   sqnorm   workspace, B*N floats (per-point |x|^2, written by the call)
 *   idx_out  (B, N, k) int32, neighbour index inside its own block;  k <= 64, k <= N
 *   dist_out optional (B, N, k) fp32 (may be NULL)                                                              */
int gfs_knn_f32(const float* x, int64_t x_bstride, int B, int C, int N, int k,
                float* sqnorm, int32_t* idx_out, float* dist_out, void* stream);

/* Same result, bit for bit, as gfs_knn_f32 (model/dgcnn.py:17-23), computed as: tcgen05 bf16-split candidate filter on
 * shifted coordinates with a per-pair error bound (two passes over the candidates: group maxima of the lower bounds give
 * the row's threshold, then the candidates whose upper bound reaches it are recorded) -> exact pinned fp32 distances of
 * the few survivors -> rank (gfs-3dseg_gws_b200/csrc/knn_tc.cu).  k <= 40, C <= 64, N <= 65535, N % 4 == 0.
 * `workspace` is scratch of gfs_knn_tc_workspace_bytes(B, C, N) bytes, 256-byte aligned (operand tiles, point-major copy,
 * per-point filter terms, up to 2 x 128 survivor records per row, repair flags); rows with more survivors than that
 * (floods of exact ties) are redone by the all-fp32 kernel inside the same call.  Four launches (prepare, filter,
 * finish, repair), no host synchronisation.  When the filter's CTA count leaves a partly empty last wave on this device
 * the blocks are processed as TWO such chains side by side (the second on an internal stream forked from and joined back
 * into `stream` with events: same stream semantics, capturable into a CUDA graph), so that one chain's finish fills the
 * SMs the other chain's filter leaves idle.  gfs_knn_tc_chains tells how many chains a call of that shape runs (1 or 2);
 * gfs_knn_tc_set_split overrides the choice: -1 automatic (default; also the GFS3D_KNN_SPLIT environment variable),
 * 0 always one chain, n > 0 the first n blocks form the first chain.  The results do not depend on it.               */
int64_t gfs_knn_tc_workspace_bytes(int B, int C, int N);
int gfs_knn_tc_chains(int B, int C, int N);
int gfs_knn_tc_set_split(int blocks_in_first_chain);
int gfs_knn_tc_f32(const float* x, int64_t x_bstride, int B, int C, int N, int k,
                   float* sqnorm, void* workspace, int64_t workspace_bytes,
                   int32_t* idx_out, float* dist_out, void* stream);
/* The neighbour SET of gfs_knn_tc_f32 / gfs_knn_f32 (the same k indices per row, in no particular order, no distances):
 * what model/dgcnn.py:118's max over the k neighbours needs.  The survivors of the filter are classified by their error
 * bounds (certainly in / certainly out / undecided) and only the undecided band gets the pinned fp32 arithmetic.       */
int gfs_knn_tc_set_f32(const float* x, int64_t x_bstride, int B, int C, int N, int k,
                       float* sqnorm, void* workspace, int64_t workspace_bytes,
                       int32_t* idx_out, void* stream);
/* Diagnostic twin (tests): additionally dumps what the tensor-core filter saw, filter_out[b][i][j] = the upper filter value
 * u ~= x~_i.x~_j - |x~_j|^2/2 + a_j on the shifted coordinates x~ (see knn_tc.cu) as (B, N, Npad) fp32 with Npad = N rounded
 * up to 256, and the per-64-row-tile repair flags (B, ceil(N/64)) int32.                                              */
int gfs_knn_tc_diag_f32(const float* x, int64_t x_bstride, int B, int C, int N, int k,
                        float* sqnorm, void* workspace, int64_t workspace_bytes,
                        int32_t* idx_out, float* filter_out, int32_t* repair_flags_out, void* stream);

/* ---- per-point fp32 1x1 conv: the split first EdgeConv conv, model/dgcnn.py:26-42 + :53 (SURVEY a3')---------
 * out[b*N+n, o] = bias[o] + sum_c x[b,c,n] * wt[c,o]        (wt = W^T, (C, O) row-major; O % 128 == 0, C <= 64)
 * For EdgeConv the caller passes wt = [s1*Wa | s1*(Wb-Wa)]^T and bias = [0 | t1] so that out = [P' | Q'].     */
int gfs_pointwise_f32(const float* x, int64_t x_bstride, int B, int C, int N,
                      const float* wt, const float* bias, int O, float* out, void* stream);

/* ---- the split first EdgeConv conv in the layout gfs_edgeconv_fwd gathers from (model/dgcnn.py:26-42 + :53, SURVEY a3')
 * wt (C, 128) = [s1*Wa | s1*(Wb-Wa)]^T, bias (128) = [0 | t1]:  P' = first 64 outputs, Q' = last 64.  Only P'[j] + Q'[i] is ever
 * used, so a per-block constant mu (the image of a point inside the block's cloud) moves from P' to Q':
 *   pb (B*N, 64) bf16 = P' - mu      (a neighbour's row: one contiguous 128-byte gather)
 *   q  (B*N, 64) fp32 = Q' + mu                                                                                      */
int gfs_edge_pq_f32(const float* x, int64_t x_bstride, int B, int C, int N, const float* wt, const float* bias,
                    void* pb, float* q, void* stream);

/* ---- fused EdgeConv given the graph: model/dgcnn.py:35-41 (gather, x_j - x_i, cat), :56-58 (LeakyReLU of conv1,
 * conv2, BN2 eval, LeakyReLU) and :118 (max over k).  h1 = LReLU(P'[j] + Q'[i]) is formed in shared memory as a
 * bf16 UMMA operand, conv2 runs on tcgen05 with the accumulator in TMEM, max over k is taken on the accumulator
 * (BN2 scale is folded into w2, so +shift and LeakyReLU commute with max) -- the (B,2C,N,k) edge tensor and the
 * (B,64,N,k) activations never exist in memory.
 *   pb, q     (B*N, 64) bf16 = P' - mu  and  (B*N, 64) fp32 = Q' + mu  from gfs_edge_pq_f32
 *   idx       (B, N, k) int32
 *   w2_packed 64x64 bf16, K-major SWIZZLE_128B image of diag(s2) W2 (gfs_pack_weight_bf16)
 *   shift2    64 floats (BN2 beta - mean*s2)
 *   y_cm      fp32 cm output, y[b, c, n] at y_cm[b*y_bstride + c*N + n], c < 64          (may be NULL)
 *   y_act     bf16 act output tile column `y_act_kb` of a matrix with y_act_kblocks 64-col blocks (may be NULL)
 *   y_act2    second optional bf16 act destination (same arguments)
 *   argmax    optional (B*N, 64) uint8: neighbour slot that produced the max (for the backward scatter)        */
int gfs_edgeconv_fwd(const void* pb, const float* q, const int32_t* idx, const void* w2_packed, const float* shift2,
                     int B, int N, int k,
                     float* y_cm, int64_t y_bstride,
                     void* y_act, int y_act_kblocks, int y_act_kb,
                     void* y_act2, int y_act2_kblocks, int y_act2_kb,
                     uint8_t* argmax, void* stream);

/* ---- weight packing for the tcgen05 kernels ---------------------------------------------------------------------
 * w (R, K) fp32 row-major, optional per-row scale (R) folded in before rounding -> bf16 tiles [ceil(K/64)][R x 64]
 * K-major SWIZZLE_128B; R % 8 == 0.  out must hold ceil(K/64)*R*128 bytes.                                        */
int gfs_pack_weight_bf16(const float* w, const float* row_scale, int R, int K, void* out, void* stream);

/* fp32 cm (B, C, N) -> bf16 act tiles (columns [kb0*64, kb0*64+C) of a matrix with kblocks blocks); C % 64 == 0 */
int gfs_cm_to_act(const float* x, int64_t x_bstride, int B, int C, int N, void* act, int kblocks, int kb0, void* stream);

/* ---- dense layer on tcgen05: Conv1d(k=1)+BN(eval)+activation, model/dgcnn.py:63-80,121-122; model/capl.py:63-65,
 * 435-457; model/attention.py:25-27 (q/k/v maps)
 * Y[m, n] = act(acc[m, n] + shift[n]),  acc = X (M x Kc, bf16 act) . Wp^T  (Wp: packed, BN scale folded, R=Nout)
 *   Nout % 16 == 0, Nout <= 256 per call;  M = B*N
 *   y_act   bf16 act destination, 64-col block offset y_kb0 in a matrix of y_kblocks blocks (may be NULL)
 *   y_cm    fp32 cm destination (B, Nout, N) with batch stride y_bstride (may be NULL)                           */
int gfs_linear_bf16(const void* x_act, int x_kblocks, int x_kb0, int kb_count,
                    const void* w_packed, const float* shift, int Nout, int act,
                    int B, int N,
                    void* y_act, int y_kblocks, int y_kb0,
                    float* y_cm, int64_t y_bstride, void* stream);

/* ---- self-attention: model/attention.py:43-46  y = softmax(q^T k * scale) v^T, flash-style on tcgen05 ----------------
 * qkv_act: bf16 act matrix holding three consecutive 64-column blocks [q | k | v] starting at block kb_q (the output of
 * one fused gfs_linear_bf16 call over the concatenated q/k/v weights).  d = 64, one head, N % 128 == 0.
 * The N x N score matrix is never written to memory.  Outputs as in gfs_edgeconv_fwd (fp32 cm and/or one bf16 act block). */
int gfs_attention_fwd(const void* qkv_act, int kblocks, int kb_q, int B, int N, float scale,
                      float* y_cm, int64_t y_bstride, void* y_act, int y_kblocks, int y_kb, void* stream);

/* ---- geometric-word projection: model/capl.py:344-353 -----------------------------------------------------------
 * cos[g] = <gp_l2[g], ec> / max(|ec|, 1e-12); cosine_feat = softmax_g(10 cos); assignment = argmax_g (first max).
 * fp32 CUDA-core contraction in a pinned order (assignment parity), fused norm/softmax/argmax.
 *   ec        cm fp32 (B, D, N), D <= 192 (batch stride ec_bstride)
 *   gp_l2t    (D, Gp) fp32: L2-normalised GW basis, transposed, zero-padded to Gp = 160 or 192 columns (G <= Gp)
 *   cosine_act bf16 act destination (G columns starting at block kb0, zero padded)    (may be NULL)
 *   cosine_cm  fp32 cm (B, G, N) destination, batch stride G*N                          (may be NULL)
 *   assignment (B*N) int32                                                                                     */
int gfs_gw_project(const float* ec, int64_t ec_bstride, int B, int D, int N,
                   const float* gp_l2t, int G, int Gp,
                   void* cosine_act, int kblocks, int kb0, float* cosine_cm, int32_t* assignment, void* stream);

/* ---- cosine / prototype logits: model/capl.py:290-322 (get_pred) fused with :127-128,:188 (get_gp_weight) -------
 * logits[b,c,n] = 10 * <proto_n[b?,c,:], feat[b,:,n]> / max(|feat|,1e-12)  [ * th if coding[c, assignment[b,n]] == 1 ]
 *   feat      cm fp32 (B, D, N), D <= 128;  proto_l2 (PB, CLS, D) already L2-normalised, PB = 1 or B;  CLS <= 32
 *   coding    optional (CLS, G) fp32 0/1 with assignment (B*N) int32 and weight th                              */
int gfs_cos_logits(const float* feat, int64_t feat_bstride, int B, int D, int N,
                   const float* proto_l2, int PB, int CLS,
                   const float* coding, int G, const int32_t* assignment, float th,
                   float* logits, void* stream);

/* ---- prototype refinement: model/capl.py:245-287 (post_refine_proto_v2), softmax over POINTS then pred @ feat^T ---
 *   logits (B, CLS, N) fp32 (= get_pred output);  feat cm (B, D, N);  out pred_proto (B, CLS, D) fp32 (un-normalised
 *   sum_n softmax_n(logits)[b,c,n] * feat[b,:,n]); the tiny gating arithmetic stays in the host wrapper.
 *   workspaces: stats (B*CLS*2) floats, partial (B * ceil(N/64) * CLS * D) floats; the reduction order is fixed.      */
int gfs_softmax_pool(const float* logits, const float* feat, int64_t feat_bstride, int B, int CLS, int D, int N,
                     float* stats, float* partial, float* pred_proto, void* stream);

/* ---- query-adaptive prototype refinement, model/capl.py:267-288 (eqn. 6) + :117-120 + the normalisation of :293 -------
 * w = max(cos(pred_proto, proto), 0);  r = w pred_proto + (1-w) proto;  base classes: r += gened; novel: r = r*0 + gened;
 * refine_l2 = r / max(|r|, 1e-12).   pred_proto (B, CLS, D), proto and gened_proto (CLS, D), refine_l2 (B, CLS, D), fp32 */
int gfs_refine_proto(const float* pred_proto, const float* proto, const float* gened_proto, int B, int CLS, int D,
                     int base_num, float* refine_l2, void* stream);

/* ---- joint histogram of two label streams: the reduction behind runs/eval.py:31-48 (evaluate_metric_GFS: confusion
 * matrix of gt x pred) and train.py:156-218 (collect_base_class_gp_coding_sum: label x geometric-word counts) ----------
 * counts[x*NB + y] += #{i : a[i] == x, b[i] == y}; points outside [0,NA) x [0,NB) are skipped (255 = ignore).
 * a, b: n int32 each, 16-byte aligned; counts: NA*NB uint64, ACCUMULATED into (the caller zeroes it); NA*NB <= 12288 */
int gfs_joint_histogram_i32(const int32_t* a, const int32_t* b, int64_t n, int NA, int NB, unsigned long long* counts,
                            void* stream);

/* ---- k-means E/M step: sklearn KMeans.fit as called at get_basis.py:210 (_k_means_lloyd.pyx:196-218) ------------
 * labels[i] = argmin_c (|c|^2 - 2 x_i.c), fp32 pinned order, strict '<' (lowest index wins).
 *   xt        (D, n) fp32: the shard's points TRANSPOSED (channel-major, like every other fp32 operand here); n % 4 == 0
 *   centers_t (D, Kp) fp32: centroids transposed, zero-padded to Kp columns (K <= Kp <= 192, Kp % 4 == 0)
 *   cnorm     workspace, Kp floats;  labels (n) int32;  score optional (n) fp32 = |c|^2 - 2 x.c of the winner          */
int gfs_kmeans_assign(const float* xt, int64_t n, int D, const float* centers_t, int K, int Kp,
                      float* cnorm, int32_t* labels, float* score, void* stream);
/* The same two results on tcgen05 (gfs-3dseg_gws_b200/csrc/rowsel_tc.cu): bf16 hi/lo split product with fp32 accumulation in
 * TMEM; rows whose best and second best score are closer than the product's error bound are re-evaluated with the pinned fp32
 * chain, so the assignment / label is the one gfs_gw_project / gfs_kmeans_assign return, bit for bit; the GW softmax features
 * (bf16 act tiles, 2e-2 tolerance) come from the tensor-core values.  D % 64 == 0, D <= 192, <= 192 entries; GW: N % 128 == 0.
 * workspace: gfs_rowsel_tc_workspace_bytes(rows, D) bytes, 256-byte aligned (packed dictionary image, re-check list).        */
int64_t gfs_rowsel_tc_workspace_bytes(int64_t rows, int D);
int gfs_gw_project_tc(const float* ec, int64_t ec_bstride, int B, int D, int N, const float* gp_l2t, int G, int Gp,
                      void* cosine_act, int kblocks, int kb0, float* cosine_cm, int32_t* assignment,
                      void* workspace, int64_t workspace_bytes, void* stream);
/* X: point_major = 0: (D, ld) channel-major as gfs_kmeans_assign takes it (ld >= n);  point_major = 1: (n, D) row-major (ld = D),
 * the layout the M-step reads -- a 128-point tile is then one contiguous piece of HBM.                                   */
int gfs_kmeans_assign_tc(const float* X, int64_t n, int64_t ld, int point_major, int D, const float* centers_t, int K, int Kp,
                         float* cnorm, int32_t* labels, void* workspace, int64_t workspace_bytes, void* stream);
/* deterministic centroid sums over X (n, D) row-major: partial (P, K, D) fp32 + pcount (P, K) int32 workspaces with
 * P = gfs_kmeans_partials() (one per SM); sums (K, D) fp64 and counts (K) int64 are reduced in a fixed order.       */
int gfs_kmeans_partials(void);
int gfs_kmeans_accumulate(const float* X, int64_t n, int D, const int32_t* labels, int K,
                          float* partial, int32_t* pcount, double* sums, int64_t* counts, void* stream);

/* The rest of a Lloyd iteration (sklearn _k_means_common.pyx:_average_centers, _kmeans.py:_kmeans_single_lloyd) in two launches:
 *   gfs_kmeans_pack:   packed (K*D + K + 1 doubles) = [sums (already there: pass packed as gfs_kmeans_accumulate's sums) |
 *                      counts as fp64 | number of i < n with labels[i] != labels_old[i]] -- the ONE buffer the sharded k-means
 *                      all-reduces per iteration.  scratch16: 16 bytes, zero on first use (the kernel leaves them zero).
 *   gfs_kmeans_update: centers_new (K, D) = count > 0 ? sums / count : 0, centers_t (D, Kp) its transpose for the next E-step,
 *                      result3 = [labels changed, sum (new - old)^2 in fp64 (fixed order), empty clusters]                 */
int gfs_kmeans_pack(const int32_t* labels, const int32_t* labels_old, int64_t n, const int64_t* counts, int K, int D,
                    double* packed, void* scratch16, void* stream);
int gfs_kmeans_update(const double* packed, const float* centers_old, int K, int D, int Kp, float* centers_new, float* centers_t,
                      double* result3, void* stream);

/* ---- k-means++ seeding step (sklearn _kmeans.py:_kmeans_plusplus behind get_basis.py:210, SURVEY 8f N3) ---------------
 * For T <= 8 candidate centres:  m[t][i] = min(max(float(|x_i|^2 - 2 x_i.c_t + |c_t|^2), 0), closest[i]),  pots[t] += sum_i m[t][i]
 * The distance is accumulated in fp64 and rounded once to fp32, as sklearn's _euclidean_distances_upcast does for float32 data.
 *   xt (D, npad) channel-major fp32 (the E-step's copy), xsq (n) fp64 squared norms, cand (T, D) row-major, closest (n) or NULL
 *   (= +inf: the first centre), m_out (T, npad) fp32, pots (T) fp64 ACCUMULATED into (the caller zeroes it)              */
int gfs_kmeans_pp_trial(const float* xt, int64_t npad, int64_t n, int D, const double* xsq, const float* cand, int T,
                        const float* closest, float* m_out, double* pots, void* stream);

/* =====================================================================================================================
 * TRAINING path (model.train(), train.py:614-631).  fp32 end to end, activations channel-major (C, M) with M = B*N points
 * or E = B*N*k edges (e = i*k + slot).  Round-1 version: correct first -- the per-edge tensors are materialised.
 * ===================================================================================================================== */

/* generic fp32 GEMM on the packed-FFMA2 core: every 1x1 conv forward (A = W^T), data gradient (A = W) and weight gradient
 * (both operands transposed, contraction over the points, split-K with a fixed-order reduction) of model/dgcnn.py:53-58,
 * 63-80 and model/capl.py:63-65,435-457; also the batched q^T k / p v products of model/attention.py:43-46.
 *   C[r, n] = bias[r] + sum_k Aop(k, r) * Bop(k, n);  Aop(k, r) = a_trans ? A[r*lda + k] : A[k*lda + r]  (B likewise with n)
 *   C stored [r*ldc + n] or, with c_trans, [n*ldc + r];  batch > 1 uses the element strides *_bstride
 *   splitk > 1 (batch == 1): workspace of splitk*R*Ncols floats; accumulate != 0 adds into C instead of overwriting      */
int gfs_gemm_f32(const float* A, int64_t lda, int a_trans, int64_t a_bstride,
                 const float* B, int64_t ldb, int b_trans, int64_t b_bstride,
                 float* C, int64_t ldc, int c_trans, int64_t c_bstride,
                 const float* bias, int R, int Ncols, int K, int batch, int splitk, float* workspace, int accumulate, void* stream);

/* the same contract on the tensor cores (csrc/gemm_tf32.cu): tcgen05.mma kind::tf32, fp32 accumulation in TMEM; operands are
 * rounded to tf32 (round-to-nearest) on their way into shared memory.
 *   split3 == 0: one product per k-step,  |C - exact| <= 2^-10 * sum_k |Aop||Bop|
 *   split3 != 0: 3xTF32 -- operands kept as hi + lo tf32 pairs, hi*hi + hi*lo + lo*hi per k-step: fp32-grade products
 *                (~1e-6); this is what the training path calls (the backward pass needs it, see the file header)        */
int gfs_gemm_tf32(const float* A, int64_t lda, int a_trans, int64_t a_bstride,
                  const float* B, int64_t ldb, int b_trans, int64_t b_bstride,
                  float* C, int64_t ldc, int c_trans, int64_t c_bstride,
                  const float* bias, int R, int Ncols, int K, int batch, int splitk, float* workspace, int accumulate, int split3,
                  void* stream);

/* BatchNorm with batch statistics (nn.BatchNorm1d/2d in training mode, model/dgcnn.py:54-55,73-74): biased variance      */
/* workspace: 2*16*C doubles (per-channel partial sums, combined in a fixed order)                                          */
int gfs_bn_stats(const float* x, int64_t ld, int C, int64_t M, double* workspace, float* mean, float* var, void* stream);
/* the same statistics plus invstd = rsqrt(var + eps), scale = gamma*invstd, shift = beta - mean*scale in the same launch       */
int gfs_bn_stats_coeffs(const float* x, int64_t ld, int C, int64_t M, double* workspace, const float* gamma, const float* beta,
                        float eps, float* mean, float* var, float* invstd, float* scale, float* shift, void* stream);
/* nn.BatchNorm running statistics, momentum form (model/dgcnn.py:54-55,73-74 under model.train()): r = (1-mom) r + mom * batch
 * with the unbiased variance var * n/(n-1); ++num_batches_tracked (int64, may be NULL)                                      */
int gfs_bn_update_running(const float* mean, const float* var, int C, int64_t n, float momentum, float* running_mean,
                          float* running_var, int64_t* num_batches_tracked, void* stream);
/* y = act(x*scale[c] + shift[c]);  act(u) = u > 0 ? u : slope*u  (0.2 LeakyReLU, 0 ReLU, 1 identity)                      */
int gfs_bn_act_fwd(const float* x, int64_t ldx, float* y, int64_t ldy, int C, int64_t M,
                   const float* scale, const float* shift, float slope, void* stream);
/* backward of y = act(gamma*xhat + beta): dx, and sum_g = dbeta, sum_gx = dgamma (per channel)                           */
int gfs_bn_act_bwd(const float* dy, int64_t lddy, const float* x, int64_t ldx, float* dx, int64_t lddx, int C, int64_t M,
                   const float* mean, const float* invstd, const float* gamma, const float* beta, float slope,
                   double* workspace, float* sum_g, float* sum_gx, void* stream);
/* the same for the BatchNorm in front of max-over-k (model/dgcnn.py:55-58,118): dy (C, Mp) is the gradient at the arg-max edge
 * arg[c, p] (< k) of every (channel, point), zero on the other edges; x and dx are the (C, Mp*k) per-edge tensors.  Replaces
 * gfs_max_over_k_bwd + gfs_bn_act_bwd without building the (C, Mp*k) gradient in between.                                   */
int gfs_bn_act_bwd_argmax(const float* dy, int64_t lddy, const uint8_t* arg, int k, const float* x, int64_t ldx, float* dx,
                          int64_t lddx, int C, int64_t Mp, const float* mean, const float* invstd, const float* gamma,
                          const float* beta, float slope, double* workspace, float* sum_g, float* sum_gx, void* stream);

/* Fusions of the per-edge BatchNorm passes of the training EdgeConv (model/dgcnn.py:53-58,118 under model.train()):
 *   gfs_bn_act_max_fwd   y[c,i] = max_slot act(z[c, i*k+slot]*scale[c] + shift[c]) and its arg-max slot, in ONE pass over z:
 *                        the (C, M*k) activated tensor of gfs_bn_act_fwd + gfs_max_over_k_fwd is never written
 *   gfs_bn_bwd_sums      the two per-channel sums of gfs_bn_act_bwd without its apply pass
 *   gfs_edge_scatter_bn  gfs_edge_scatter of dH = BN/activation backward of (dy = d h1, x = H), computed while the tile is staged:
 *                        the (64, E) tensor dH is never written or re-read                                                    */
int gfs_bn_act_max_fwd(const float* z, int C, int64_t M, int k, const float* scale, const float* shift, float slope, float* y,
                       int64_t ldy, uint8_t* arg, void* stream);
int gfs_bn_bwd_sums(const float* dy, int64_t lddy, const float* x, int64_t ldx, int C, int64_t M, const float* mean,
                    const float* invstd, const float* gamma, const float* beta, float slope, double* workspace, float* sum_g,
                    float* sum_gx, void* stream);
int gfs_edge_scatter_bn(const float* dy, const float* x, const int32_t* idx, int B, int N, int k, const float* mean,
                        const float* invstd, const float* gamma, const float* beta, float slope, const float* sum_g,
                        const float* sum_gx, float* dpq, void* stream);

/* Deterministic variant of gfs_edge_scatter_bn: the backward of the neighbour gather of model/dgcnn.py:38-41 summed in a fixed order.
 * Edge e = i*k + slot of point i (block b = i / N) targets j = b*N + idx[e]; idx values lie in [0, N).
 *   gfs_edge_reverse_index       CSR of the incoming edges, identical to a stable sort of the targets: rev_ptr (B*N + 1 int32)
 *                                holds the exclusive scan of the in-degrees, rev_edge (E = B*N*k int32) the edges of each target in
 *                                ascending edge index.  Built without order-dependent atomics: the same on every run.
 *                                N <= 57 856 (per-target counters in shared memory).
 *   gfs_edge_scatter_bn_ordered  dpq (M, 128), every element written (no zeroing needed).  Q half (c >= 64): exactly as
 *                                gfs_edge_scatter_bn.  P half: dpq[j, c] = fp32 sum, left to right from +0.0, of t[e, c] over the
 *                                edges of target j in ascending edge index (a target without incoming edges gets +0.0), where
 *                                t[e, c] is the per-edge BatchNorm / activation backward term gfs_edge_scatter_bn adds.  The terms
 *                                are first stored to edge_terms (E x 64 fp32, caller-owned, 16-byte aligned), then summed per target.
 * Both reject k > 64 and E >= 2^31 with GFS_ERR_UNSUPPORTED.                                                                      */
int gfs_edge_reverse_index(const int32_t* idx, int B, int N, int k, int32_t* rev_ptr, int32_t* rev_edge, void* stream);
int gfs_edge_scatter_bn_ordered(const float* dy, const float* x, const int32_t* idx, const int32_t* rev_ptr, const int32_t* rev_edge,
                                int B, int N, int k, const float* mean, const float* invstd, const float* gamma, const float* beta,
                                float slope, const float* sum_g, const float* sum_gx, float* edge_terms, float* dpq, void* stream);

/* edge tensor of model/dgcnn.py:35-41 after the split first conv: H[c, e] = P[j(e), c] + Q[i(e), c]  (pq point-major (M,128)) */
int gfs_edge_gather(const float* pq, const int32_t* idx, int B, int N, int k, float* H, void* stream);
/* the same plus the batch statistics of H and the BatchNorm coefficients (as gfs_bn_stats_coeffs) taken while the tiles are on
 * chip: no second pass over H.  partials: 64 * 2 * ceil(E/128) float pairs (sum, sum of squares), reduced in fp64 in a fixed order */
int gfs_edge_gather_stats(const float* pq, const int32_t* idx, int B, int N, int k, float* H, float* partials,
                          const float* gamma, const float* beta, float eps, float* mean, float* var, float* invstd,
                          float* scale, float* shift, void* stream);
/* its backward: dP[j] += dH[:, e], dQ[i] += dH[:, e]  (dpq (M,128) must be zeroed by the caller; fp32 atomics)            */
int gfs_edge_scatter(const float* dH, const int32_t* idx, int B, int N, int k, float* dpq, void* stream);
/* model/dgcnn.py:118: y[c, i] = max over the k slots of a[c, i*k + slot] (first maximum) + arg-max slot; and its backward  */
int gfs_max_over_k_fwd(const float* a, int C, int64_t M, int k, float* y, int64_t ldy, uint8_t* arg, void* stream);
int gfs_max_over_k_bwd(const float* dy, int64_t lddy, const uint8_t* arg, int C, int64_t M, int k, float* da, void* stream);
/* model/attention.py:45: p0 = softmax(s*scale) per row, p = p0 * dropout; backward.  The dropout factor (1/keep or 0) comes from
 * an explicit mask (rows x n floats), or -- mask == NULL and keep < 1 -- from a counter-based hash of (seed, row, column) that
 * the backward regenerates, so no mask tensor exists; keep >= 1 and mask == NULL: no dropout (p may alias p0).
 * gfs_dropout_mask materialises the hash's mask (tests).                                                                     */
int gfs_softmax_rows_fwd(const float* s, int64_t rows, int n, float scale, const float* mask, uint32_t seed, float keep,
                         float* p0, float* p, void* stream);
int gfs_softmax_rows_bwd(const float* p0, const float* dp, const float* mask, uint32_t seed, float keep, int64_t rows, int n,
                         float scale, float* ds, void* stream);
int gfs_dropout_mask(int64_t rows, int n, uint32_t seed, float keep, float* mask, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GFS3D_H */
