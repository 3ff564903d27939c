/*
 * ev2h.h - C ABI of libev2h.so: the Ev2Hands set-abstraction encoder hot path
 * as hand-written sm_100a CUDA kernels.
 *
 * The reference has no FFI for this path: it is pure PyTorch in
 * src/Ev2Hands/model/pointnet2_utils.py and the drop-in boundary is that
 * module's Python namespace (imported at src/Ev2Hands/model/TEHNet.py:6).
 * Each entry point below names the reference function it replaces; the Python
 * side (ev2hands_b200/pointnet2_utils.py) re-creates the reference's classes on
 * top of these calls, and INTEGRATION.md shows the one-line change that makes
 * TEHNet.py use them.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  Every pointer is DEVICE
 *     memory unless the name ends in _host.
 *   - the caller owns every buffer, including scratch; the library allocates
 *     nothing on the device and keeps no mutable global state, so it may be
 *     called from one host thread per GPU (nn.DataParallel, train.py:68).
 *   - kernels are enqueued on `stream` (a cudaStream_t) of the current device
 *     and the call returns without synchronising.
 *   - return value: 0 on success, otherwise an ev2h_status; the message for the
 *     calling thread is available from ev2h_last_error().  Nothing throws.
 *   - index outputs are int32 (the reference uses int64; the Python wrappers
 *     widen them where the reference API hands indices to the user).
 *   - "cf" = channel-first  [B, C, N]  (how the model passes tensors around),
 *     "rows" = point-major  [B, N, C]  (how the kernels gather).
 */
#ifndef EV2H_H
#define EV2H_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *ev2h_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define EV2H_API __attribute__((visibility("default")))
#else
#define EV2H_API
#endif

typedef enum {
    EV2H_OK = 0,
    EV2H_ERR_BAD_ARGUMENT = 1,  /* null pointer, non-positive size, misaligned buffer */
    EV2H_ERR_UNSUPPORTED = 2,   /* shape outside what the kernels are built for */
    EV2H_ERR_CUDA = 3,          /* a CUDA runtime call or launch failed */
    EV2H_ERR_WORKSPACE = 4      /* scratch buffer too small */
} ev2h_status;

/* Library version, and the message attached to the last non-zero status
 * returned on the calling thread ("" if none). */
EV2H_API int ev2h_version(void);
EV2H_API const char *ev2h_last_error(void);

/* ---- farthest point sampling -------------------------------------------------
 * Replaces farthest_point_sample (pointnet2_utils.py:63-84) followed by
 * index_points(xyz, fps_idx) (pointnet2_utils.py:239).
 * xyz is read in place from a channel-first tensor through element strides, so
 * the non-contiguous view xyz[:, :3, :] of TEHNet.py:174 needs no copy:
 *   x_c(b, n) = xyz[b*stride_b + c*stride_c + n*stride_n],  c = 0..2.
 * start_idx[b] is the first sample (the reference draws it with torch.randint on
 * the CPU generator, pointnet2_utils.py:75; the caller draws it the same way).
 * Outputs (any may be NULL): idx int32 [B,S]; centres as rows [B,S,3] and as
 * channel-first [B,3,S].  Bit-exact with the reference: distances are
 * (dx*dx + dy*dy) + dz*dz with every product and sum rounded separately, and
 * ties go to the lowest index.  Limits: 1 <= S, 1 <= N <= 16384. */
EV2H_API int ev2h_fps_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                 const int64_t *start_idx, int B, int N, int S,
                 int32_t *out_idx, float *out_centres_rows, float *out_centres_cf,
                 ev2h_stream_t stream);
/* ev2h_fps_f32 with the kernel for long windows (4096 < N <= 16384) chosen by the caller: 1 = exhaustive single CTA,
 * 2 = one thread-block cluster per window (distributed shared memory), 3 = spatially pruned (points bucketed by Morton
 * cell; a bucket whose bounding box is at least as far from the new centre as its largest running minimum is skipped -
 * exact, because the bound uses the point distance's own rounding sequence); 0 = the library's choice (2 while N > 8192
 * and every cluster is resident at once, else 3).  Every variant
 * returns the same bits; the entry exists for the tests that prove it and for measurements.  N <= 4096: variant ignored. */
EV2H_API int ev2h_fps_variant_f32(int variant, const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                  const int64_t *start_idx, int B, int N, int S, int32_t *out_idx,
                                  float *out_centres_rows, float *out_centres_cf, ev2h_stream_t stream);

/* ---- multi-radius ball query --------------------------------------------------
 * Replaces query_ball_point (pointnet2_utils.py:87-107) for every radius of a
 * multi-scale layer in one pass over the points, and with it square_distance
 * (pointnet2_utils.py:19-40): the distance is evaluated in the reference's
 * expanded form -2*(q.p) + |q|^2 + |p|^2 with its roundings (dot product as an
 * FMA chain x,y,z; norms as (x*x + y*y) + z*z; the two adds one after the
 * other), and a point is kept when NOT (d > radius_sq[i]).
 * radius_sq_host[i] = (float)(radius_i * radius_i evaluated in double), which is
 * what aten compares against.  nsample_host[i] = K_i.
 * out_idx int32 [B, S, sum_i K_i]: for centre s the K_0 slots of scale 0, then
 * the K_1 slots of scale 1, ...; each block holds the first K_i in-radius point
 * indices in ascending order, padded with the first one; if no point is in
 * radius every slot holds N (the reference's sentinel).
 * Limits: n_scales <= 4, N <= 65536. */
EV2H_API int ev2h_ball_query_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                        const float *centres_rows, int B, int N, int S,
                        int n_scales, const float *radius_sq_host, const int32_t *nsample_host,
                        int32_t *out_idx, ev2h_stream_t stream);

/* The same query that also reports, per centre and scale, how many of the K slots hold real
 * (unpadded) neighbours: out_cnt int32 [n_scales, B, S] (scale-major), 0 when no point is in radius. */
EV2H_API int ev2h_ball_query_cnt_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                        const float *centres_rows, int B, int N, int S,
                        int n_scales, const float *radius_sq_host, const int32_t *nsample_host,
                        int32_t *out_idx, int32_t *out_cnt, ev2h_stream_t stream);

/* first[b,n] = 1 iff no point m < n of window b has the same 32-byte record pts8[b,m,:] (bitwise).  Event
 * windows are sampled with replacement, so ~40 % of the points are exact copies of an earlier one; copies give
 * identical MLP rows and the compacted row list keeps only the first.  N <= 16384 (an open-addressing table of the
 * next power of two >= 2 N slots in shared memory). */
EV2H_API int ev2h_first_occurrence_u8(const float *pts8, int B, int N, uint8_t *first, ev2h_stream_t stream);
/* Ball query that also emits, per centre and scale, the first-K hit list WITHOUT the hits whose first flag is 0
 * (out_uniq int32 [B,S,sum K], only the first out_ucnt[scale,b,s] entries of each block are written;
 * out_ucnt int32 [n_scales,B,S]).  out_idx is the reference's padded list as in ev2h_ball_query_f32. */
EV2H_API int ev2h_ball_query_uniq_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                        const float *centres_rows, int B, int N, int S,
                        int n_scales, const float *radius_sq_host, const int32_t *nsample_host,
                        int32_t *out_idx, const uint8_t *first_flag, int32_t *out_uniq, int32_t *out_ucnt,
                        ev2h_stream_t stream);

/* Ball query with the row compaction of ev2h_group_compact_i32 done in the same kernel (no second pass over the
 * index lists): out_idx as in ev2h_ball_query_f32, plus rowmap / blockgroup / n_rows as described below.
 * first_flag (optional, with uniq_scratch int32 [B,S,sum K]) also drops exact-duplicate points. */
EV2H_API int ev2h_ball_query_compact_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                        const float *centres_rows, int B, int N, int S,
                        int n_scales, const float *radius_sq_host, const int32_t *nsample_host,
                        int32_t *out_idx, const uint8_t *first_flag, int32_t *uniq_scratch,
                        int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                        ev2h_stream_t stream);

/* Row compaction for the fused kernel.  query_ball_point pads every group to K neighbours with copies of
 * the first one (pointnet2_utils.py:104-106); the max-pool cannot see those copies, so the shared MLP need
 * not evaluate them.  For every scale i of a layer this builds the list of rows actually needed - per group
 * its out_cnt real neighbours, rounded up to a multiple of 8 with copies of the first, groups back to back:
 *   rowmap_host[i]      int32 [B*S*K_i]        global point row b*N + point of every compact row (-1: no point)
 *   blockgroup_host[i]  int32 [B*S*K_i/8]      global group b*S + centre of every 8-row block
 *   n_rows_dev          int32 [n_scales]       compact rows per scale
 * (device buffers; the two pointer tables live on the host).  Groups are appended in no particular order
 * (one atomic add per group reserves its rows); nothing downstream depends on the order.
 * idx / cnt come from ev2h_ball_query_cnt_f32, or (out_uniq, out_ucnt) from ev2h_ball_query_uniq_f32 to drop
 * exact-duplicate points as well; every K_i must be a multiple of 8. */
EV2H_API int ev2h_group_compact_i32(const int32_t *idx, int idx_ld, const int32_t *cnt, int B, int N, int S, int n_scales,
                                    const int32_t *nsample_host,
                                    int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                                    ev2h_stream_t stream);

/* square_distance as a standalone op (pointnet2_utils.py:19-40), same arithmetic as
 * inside the ball query: src_rows [B,S,3], dst_rows [B,N,3] -> out [B,S,N]. */
EV2H_API int ev2h_square_distance_f32(const float *src_rows, const float *dst_rows, int B, int S, int N,
                             float *out, ev2h_stream_t stream);

/* index_points (pointnet2_utils.py:43-60): out[b,m,:] = table_rows[b, idx[b,m], :],
 * table_rows [B,N,C], idx int32 [B,M] (any trailing shape flattened into M). */
EV2H_API int ev2h_index_rows_f32(const float *table_rows, const int32_t *idx, int B, int N, int M, int C,
                        float *out, ev2h_stream_t stream);

/* ---- grouping (materialising gather) -------------------------------------------
 * Replaces the index_points / subtract / cat sequence of
 * PointNetSetAbstractionMsg.forward (pointnet2_utils.py:244-248):
 *   row (b, s, j) = [ feats_rows[b, p, 0..D) , xyz(b, p) - centre(b, s) , 0-pad ]
 * with p = idx[b, s, k_off + j], j < K.  feats_rows may be NULL (D = 0).
 * out is [B*S*K, ld_out] f32 with ld_out >= D + 3; columns past D+3 are zeroed.
 * idx has row length idx_ld (= sum K_i) so one scale is selected by k_off. */
EV2H_API int ev2h_group_gather_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                          const float *feats_rows, int D, const float *centres_rows,
                          const int32_t *idx, int idx_ld, int k_off,
                          int B, int N, int S, int K, float *out, int ld_out,
                          ev2h_stream_t stream);

/* Backward of the feature part of the gather (autograd of index_points,
 * pointnet2_utils.py:43-60): grad_feats_rows[b, p, :] += grad_rows[(b,s,j), 0..D)
 * for p = idx[b,s,k_off+j].  grad_feats_rows [B,N,D] must be zeroed by the
 * caller (or hold the sum so far, e.g. from another scale). */
EV2H_API int ev2h_group_gather_bwd_f32(const float *grad_rows, int ld_grad, const int32_t *idx, int idx_ld,
                              int k_off, int B, int N, int S, int K, int D,
                              float *grad_feats_rows, ev2h_stream_t stream);

/* ---- 32-byte point records for the gather mode of the fused kernel -----------------------------
 * pts8[b, n, :] = [feats[b, 0..D, n] | xyz[b, 0..3, n] | 0 ...] from two channel-first tensors read through element
 * strides (the reference's points [B, D, N] and xyz = points[:, :3, :], TEHNet.py:172-175); D + 3 <= 8, feats may be
 * NULL with D = 0.  One record = one 32-byte sector per gathered neighbour. */
EV2H_API int ev2h_point_records_f32(const float *feats, int64_t feats_stride_b, int64_t feats_stride_c, int64_t feats_stride_n, int D,
                                    const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                    int B, int N, float *pts8, ev2h_stream_t stream);

/* ---- batched transpose between the two layouts ----------------------------------
 * dst[b*dst_stride_b + c*dst_ld + dst_col_off + r] = src[b*src_stride_b + r*src_stride_r + c*src_stride_c]
 * for r < R, c < C.  Used for cf -> rows (permute(0,2,1).contiguous(),
 * pointnet2_utils.py:233-235) and rows -> cf on the way out, and to lay xyz and
 * features side by side for sample_and_group_all (pointnet2_utils.py:141-158). */
EV2H_API int ev2h_transpose_f32(const float *src, int64_t src_stride_b, int64_t src_stride_r, int64_t src_stride_c,
                       int B, int R, int C, float *dst, int64_t dst_stride_b, int64_t dst_ld,
                       int64_t dst_col_off, ev2h_stream_t stream);

/* ---- weight preparation -----------------------------------------------------------
 * Folds a 1x1 convolution's bias and an eval-mode BatchNorm into one affine map
 * (Conv2d + BatchNorm2d pairs of pointnet2_utils.py:167-173, :210-222):
 *   scale = gamma / sqrt(var + eps);  W' = scale * W;  b' = scale * (b - mean) + beta
 * conv_w is [Cout, Cin].  Output layout for the fp32 kernels: wt is
 * [Cin_pad, Cout_pad] (input channel major, zero padded; Cin_pad = roundup(Cin,16),
 * Cout_pad = roundup(Cout,128)), bias_out is [Cout_pad]. */
EV2H_API int ev2h_fold_conv_bn_f32(const float *conv_w, const float *conv_b, const float *bn_gamma,
                          const float *bn_beta, const float *bn_mean, const float *bn_var, double eps,
                          int Cin, int Cout, float *wt, float *bias_out,
                          ev2h_stream_t stream);

/* ---- shared MLP layer on CUDA cores, fp32 ------------------------------------------
 * One 1x1-conv + folded BN + ReLU layer over M rows (pointnet2_utils.py:253-256):
 *   y[m, 0..Cout) = relu( x[m, 0..Cin) . W' + b' )
 * x is [M, ld_x] (ld_x % 4 == 0, 16-byte aligned; columns Cin .. ld_x - 1 are padding
 * and never enter the product, whatever they hold), wt/bias come from
 * ev2h_fold_conv_bn_f32.  pool_rows == 0: y is [M, ld_y].  pool_rows = K > 0 fuses
 * the max over each run of K consecutive rows (torch.max(x, 2)[0],
 * pointnet2_utils.py:257): y is [M/K, ld_y] written at column y_col_off and MUST be
 * zero-filled by the caller beforehand (post-ReLU values are >= 0).  y needs only the
 * alignment of a float.
 * argmax (optional, only with pool_rows) is not produced here; see
 * ev2h_group_max_f32 for the training path. */
EV2H_API int ev2h_linear_relu_f32(const float *x, int64_t M, int ld_x, int Cin, const float *wt,
                         const float *bias, int Cout, int pool_rows, float *y, int ld_y,
                         int y_col_off, ev2h_stream_t stream);

/* The same layer without the ReLU: y = x W' + b' (no pooling).  Used to evaluate a layer's
 * linear part once per point when it commutes with the grouping (see ev2h_sa_msg_fused_tc). */
EV2H_API int ev2h_linear_f32(const float *x, int64_t M, int ld_x, int Cin, const float *wt, const float *bias,
                             int Cout, float *y, int ld_y, int y_col_off, ev2h_stream_t stream);

/* ---- shared MLP layer on the tensor cores (tcgen05 / TMEM) ----------------------------
 * Same contract as ev2h_linear_relu_f32 (x, y fp32 in HBM; bias from ev2h_fold_conv_bn_f32)
 * with the contraction on the 5th-generation tensor cores.  mode selects the arithmetic:
 *   EV2H_TC_BF16   (0)  operands rounded to bf16, fp32 accumulate  (feature bar 1e-2)
 *   EV2H_TC_TF32X3 (1)  error-compensated split x = hi + lo, w = hi + lo, three tf32 products,
 *                       fp32 accumulate: fp32-level accuracy     (feature bar 1e-5)
 *   EV2H_TC_TF32_BF16C (2)  the same split with hi*hi in tf32 and the two correction products
 *                       x_lo*w_hi + x_hi*w_lo on bf16 copies (their 2^-9 rounding is 2^-20 of the result):
 *                       fp32-level accuracy at two thirds of the tensor work (feature bar 1e-5).
 *                       Accepted by ev2h_sa_msg_fused_tc and by ev2h_tc_pack_weights_kc for its weights.
 * Weights must first be packed from the folded layout (wt, ld_w = round_up(Cout,128) as
 * written by ev2h_fold_conv_bn_f32) into the kernel's shared-memory image:
 * ev2h_tc_packed_bytes gives the buffer size, ev2h_tc_pack_weights fills it.
 * pool_rows must be 0, 32, 64 or a multiple of 128; Cout <= 256 or a multiple of 256;
 * other shapes return EV2H_ERR_UNSUPPORTED (callers use ev2h_linear_relu_f32 for those).
 * Columns Cin .. ld_x - 1 of x are padding and never enter the product, whatever they hold (NaN included).
 * Output columns: without pooling (pool_rows == 0, ev2h_linear_tc, ev2h_conv1d_tc) the kernel writes columns
 * y_col_off .. y_col_off + P - 1 of every row, where P = min(ld_y - y_col_off, Cout rounded up to the accumulator
 * block: a multiple of 16 below 256 channels, of 256 above): the Cout results, then exact +0.0 in the padding
 * columns.  A caller sizing rows to round_up(Cout, 4) gets those padding columns zeroed.  With pooling only the
 * Cout result columns of each pooled row are written.  Every other column of y keeps what it held.
 * x and w_packed must be 16-byte aligned; y needs only the alignment of a float.
 * range_flag (device int32, may be NULL; used with EV2H_TC_F16X3 only): bit 0 is set (atomic OR, never
 * cleared) when an input operand left the fp16 range (|x| >= 65520) or was NaN.  The caller also checks the
 * weights it packs: the kernels see them only as fp16 pairs. */
#define EV2H_TC_BF16 0
#define EV2H_TC_TF32X3 1
#define EV2H_TC_TF32_BF16C 2
#define EV2H_TC_F16X3 3      /* x = hi + lo, w = hi + lo as fp16 pairs, three kind::f16 products: fp32-level accuracy for
                              * |operands| < 65520; an activation outside that range (or NaN) raises the range_flag
                              * of every entry that takes one (per-layer and fused kernels) */
EV2H_API int64_t ev2h_tc_packed_bytes(int Cin, int Cout, int mode);
EV2H_API int ev2h_tc_pack_weights(const float *wt, int ld_w, int Cin, int Cout, int mode, void *packed,
                                  ev2h_stream_t stream);
/* The tensor-core layer without the ReLU (y = x W' + b'), cf. ev2h_linear_f32. */
EV2H_API int ev2h_linear_tc(const float *x, int64_t M, int ld_x, int Cin, const void *w_packed, const float *bias,
                            int Cout, float *y, int ld_y, int y_col_off, int mode, int32_t *range_flag,
                            ev2h_stream_t stream);

/* Same with an explicit K-chunk length (16 or 32 input channels per shared-memory image;
 * ev2h_sa_msg_fused_kc tells which one the fused kernel wants) and row padding of the image:
 * row_align 16 when the weights are the UMMA B operand, 128 when they are the A operand (the
 * fused kernel's last layer, whose output channels are the accumulator's TMEM lanes). */
EV2H_API int64_t ev2h_tc_packed_bytes_kc(int Cin, int Cout, int mode, int kc, int row_align);
EV2H_API int ev2h_tc_pack_weights_kc(const float *wt, int ld_w, int Cin, int Cout, int mode, int kc, int row_align,
                                     void *packed, ev2h_stream_t stream);
EV2H_API int ev2h_linear_relu_tc(const float *x, int64_t M, int ld_x, int Cin, const void *w_packed,
                                 const float *bias, int Cout, int pool_rows, float *y, int ld_y,
                                 int y_col_off, int mode, int32_t *range_flag, ev2h_stream_t stream);
/* ---- weight gradient of a 1x1 convolution over point rows (training path) ---------------------------------
 * dW [Cout, Cin] (row-major, contiguous) = dY^T X with dY [M, ld_dy >= Cout] and X [M, ld_x >= Cin] fp32 rows - the
 * autograd of Conv2d(1x1) (pointnet2_utils.py:253-256) when the grouped tensor is kept as rows: a GEMM whose contraction
 * runs over the M = B*S*K rows.  Slabs of rows are accumulated with exact fp32 FMAs and summed in a fixed order
 * (deterministic).  db [Cout] (optional, may be NULL) = the column sums of dY, the bias gradient, accumulated in the same
 * pass.  workspace: ev2h_wgrad_splits(M, Cout, Cin) * Cout * (Cin + 1) floats. */
EV2H_API int ev2h_wgrad_splits(int64_t M, int Cout, int Cin);
EV2H_API int ev2h_wgrad_f32(const float *dy, int ld_dy, const float *x, int ld_x, int64_t M, int Cout, int Cin,
                            float *workspace, float *dw, float *db, ev2h_stream_t stream);

/* ---- sampling and ball query in ranges (front-end pipelining) ---------------------------------------
 * The S iterations of farthest_point_sample are strictly sequential (pointnet2_utils.py:76-83) and only B CTAs wide,
 * but the ball query of centre s needs nothing of the centres after it.  ev2h_fps_range_f32 runs samples
 * [s_begin, s_end) of S and carries the running minimum distances / the next centre to the following call through
 * state_best [B, N] fp32 / state_cur [B] int32 (written when s_end < S, read when s_begin > 0); the outputs are the
 * same arrays ev2h_fps_f32 writes, bit for bit.  ev2h_ball_query_compact_range_f32 is ev2h_ball_query_compact_f32 for
 * the centres [s_begin, s_begin + s_count) only (s_begin a multiple of 32); reset_rows = 0 keeps appending to the
 * compacted row lists of an earlier range.  Issued on two streams, the ball query of one range runs beside the
 * sampling of the next.  N <= 4096. */
EV2H_API int ev2h_fps_range_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                const int64_t *start_idx, int B, int N, int S, int s_begin, int s_end,
                                float *state_best, int32_t *state_cur, int32_t *out_idx,
                                float *out_centres_rows, float *out_centres_cf, ev2h_stream_t stream);
EV2H_API int ev2h_ball_query_compact_range_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                               const float *centres_rows, int B, int N, int S, int s_begin, int s_count,
                                               int reset_rows, int n_scales, const float *radius_sq_host,
                                               const int32_t *nsample_host, int32_t *out_idx, const uint8_t *first_flag,
                                               int32_t *uniq_scratch, int32_t *const *rowmap_host,
                                               int32_t *const *blockgroup_host, int32_t *n_rows_dev, ev2h_stream_t stream);

/* ---- Conv1d over rows on the tensor cores (SURVEY.md 8f row N2) ---------------------------------
 * Replaces nn.Conv1d(Cin, Cout, kernel_size = taps, stride 1, padding = taps / 2) [+ ReLU] [+ BatchNorm1d (eval)
 * AFTER the ReLU] of the segmentation classifier and the per-hand query convolutions (reference TEHNet.py:135-166,
 * applied at :188-192) on point-major rows: x_rows [M, ld_x] holds M / rows_per_seq sequences of rows_per_seq
 * positions x Cin channels; y[r] = act(sum_t W_t x[r + t - taps/2] + b) * post_scale + post_shift, rows outside a
 * sequence counting as zero (the convolution's zero padding).  The shifted rows are gathered by the kernel's loaders;
 * no im2col buffer exists.  w_packed = ev2h_tc_pack_weights_kc image of the [taps * Cin, Cout] matrix whose row
 * t * Cin + ci is W[:, ci, t] (kc 32, row_align 16); post_scale / post_shift may be NULL.  taps in {1, 3, 5}.
 * Columns Cin .. ld_x - 1 of x_rows are padding and never enter the product; range_flag, the output columns written
 * (the Cout results plus exact-zero padding up to the accumulator block width) and the alignment rules as for
 * ev2h_linear_tc. */
EV2H_API int ev2h_conv1d_tc(const float *x_rows, int64_t M, int ld_x, int Cin, int taps, int rows_per_seq, const void *w_packed,
                            const float *bias, int Cout, int relu, const float *post_scale, const float *post_shift,
                            float *y, int ld_y, int y_col_off, int mode, int32_t *range_flag, ev2h_stream_t stream);

/* ---- class-wise attention pooling (SURVEY.md 8f row N2) ------------------------------------------
 * Replaces AttentionBlock.forward (reference TEHNet.py:9-27): sim[b,c,d] = scale * sum_n key[b,n,c] query[b,n,d],
 * softmax over the C classes, context[b,c,n] = sum_d softmax[b,c,d] value[b,n,d].  Rows are point-major:
 * key_rows [B*N, ld_k] (C <= 8 columns), query_rows [B*N, ld_q], value_rows [B*N, ld_v] (D columns, D % 32 == 0,
 * D <= 1024); partial [B, 8, C, D] fp32 workspace; out_cf [B, C, N] channel-first, the layout the hand regressor's
 * set abstraction takes its features in (TEHNet.py:194-195).  Deterministic (fixed summation order), exact fp32. */
EV2H_API int ev2h_class_attention_f32(const float *key_rows, int ld_k, const float *query_rows, int ld_q,
                                      const float *value_rows, int ld_v, int B, int N, int C, int D, float scale,
                                      float *partial, float *out_cf, ev2h_stream_t stream);

/* ---- fused grouping + shared MLP + max-pool for ONE radius scale (tensor cores) ------------
 * Replaces the body of the per-radius loop of PointNetSetAbstractionMsg.forward
 * (pointnet2_utils.py:243-257): gather of the K neighbours of every centre, the three
 * Conv2d(1x1)+BatchNorm2d(eval)+ReLU layers and the max over K, without materialising the
 * grouped tensor or any intermediate activation in HBM.
 *   idx [B,S,idx_ld] int32 from ev2h_ball_query_f32, this scale's K slots start at k_off;
 *   centres_rows [B,S,3];  K in {32, 64, 128};  every layer width <= 256.
 * Layer 1 (width c1), one of:
 *   gather mode    (P == NULL): pts8 [B,N,8] rows = [features(D) | xyz | 0], D + 3 <= 8; the kernel
 *                  forms [features | xyz - centre] as the reference does and evaluates layer 1 in
 *                  exact fp32 on the CUDA cores from first_wt_host / first_bias_host: HOST copies of
 *                  the folded map written by ev2h_fold_conv_bn_f32 (row length first_ld, c1 <= 128).
 *                  They travel as kernel parameters (constant bank), which keeps the loaders'
 *                  weight reads off the shared-memory pipe the tensor cores' operands saturate.
 *   per-point mode (P != NULL): layer 1 was evaluated per point / per centre:
 *                  P [B*N, ld_p] = W1' [features; xyz] + b1' (ev2h_linear_f32) at column p_col,
 *                  C [B*S, ld_c] = W1'_xyz centre at column c_col; the kernel forms
 *                  relu(P[point] - C[centre]); c1 must be a multiple of 32.
 * Layers 2 and 3 run on the tensor cores: cout_host[2] their widths, w_packed_host[2] their
 * ev2h_tc_pack_weights_kc images (kc from ev2h_sa_msg_fused_kc), bias_host[2] their folded biases
 * (device pointers in host arrays).  out_rows [B*S, ld_out]: the pooled features of this scale
 * are written at column out_col.  mode: EV2H_TC_BF16 / EV2H_TC_TF32X3 / EV2H_TC_TF32_BF16C / EV2H_TC_F16X3.
 * range_flag (device int32, may be NULL): bit 0 is set when an EV2H_TC_F16X3 activation operand left the fp16
 * range or was NaN (the layer-1 outputs and the layer-2 activations the kernel splits itself).
 * Deviation from the reference (all modes): ReLU and the max-pool are evaluated with fmaxf / an integer atomic
 * max on zero-initialised output, so a NaN activation becomes 0 where F.relu / torch.max would propagate it. */
EV2H_API int ev2h_sa_msg_fused_tc(
    const int32_t *idx, int idx_ld, int k_off, const float *centres_rows, int B, int N, int S, int K,
    const float *pts8, int D, const float *first_wt_host, int first_ld, const float *first_bias_host,
    const float *P, int ld_p, int p_col, const float *C, int ld_c, int c_col,
    int c1, const int32_t *cout_host, const void *const *w_packed_host, const float *const *bias_host,
    float *out_rows, int ld_out, int out_col, int mode, int32_t *range_flag, ev2h_stream_t stream);

/* The fused kernel over a compacted row list (ev2h_group_compact_i32) instead of the dense [B,S,K] index
 * block: same arguments otherwise, bit-identical pooled features (out_rows must be zero-filled: groups that
 * straddle two row tiles are merged with an atomic max), time proportional to the real neighbours. */
EV2H_API int ev2h_sa_msg_fused_compact_tc(
    const int32_t *rowmap, const int32_t *blockgroup, const int32_t *n_rows_dev,
    const float *centres_rows, int B, int N, int S, int K,
    const float *pts8, int D, const float *first_wt_host, int first_ld, const float *first_bias_host,
    const float *P, int ld_p, int p_col, const float *C, int ld_c, int c_col,
    int c1, const int32_t *cout_host, const void *const *w_packed_host, const float *const *bias_host,
    float *out_rows, int ld_out, int out_col, int mode, int32_t *range_flag, ev2h_stream_t stream);

/* K-chunk length (16 or 32) the fused kernel uses for layers of widths cout_host[2], i.e. the kc
 * to pack their weights with; -1 if the pair is not supported. */
EV2H_API int ev2h_sa_msg_fused_kc(int mode, const int32_t *cout_host);

/* Debug/profiling only: device buffer of 512 x 16 int64 receiving the timeline trace of CTA 0 of the next fused
 * launches (only in builds with -DEV2H_FUSED_TRACE, see tools/fused_trace.py; NULL turns it off). */
EV2H_API int ev2h_fused_set_debug_buffer(void *buf);
/* Debug only: bit 0 swaps the leading/stride byte offsets of the UMMA shared-memory descriptors. */
EV2H_API int ev2h_tc_set_debug(int flags);

/* ---- max-pool over the neighbour axis, with argmax, and its backward -----------------
 * Training path (BatchNorm in batch-statistics mode keeps conv/BN/ReLU in
 * PyTorch; see DESIGN.md).  x is channel-first [B, C, K, S] as the reference's
 * convolutions produce it (pointnet2_utils.py:252); out [B, C, S]; arg int32
 * [B, C, S] = first k attaining the max (torch.max's tie-break on CUDA and CPU).
 * Backward routes grad_out to x[b, c, arg, s] and writes zeros elsewhere. */
EV2H_API int ev2h_group_max_f32(const float *x, int B, int C, int K, int S, float *out, int32_t *arg,
                       ev2h_stream_t stream);
EV2H_API int ev2h_group_max_bwd_f32(const float *grad_out, const int32_t *arg, int B, int C, int K, int S,
                           float *grad_x, ev2h_stream_t stream);

/* ---- feature propagation (decoder; SURVEY.md section 8f row N1) -------------------------
 * Replaces the geometric half of PointNetFeaturePropagation.forward (pointnet2_utils.py:294-301):
 * square_distance(xyz1, xyz2), the full sort of every row, the first three, and
 * weight = (1 / (d + 1e-8)) / sum.  xyz1 (queries, N per window) and xyz2 (sources, S >= 3 per
 * window) are channel-first [B,3,*] addressed through element strides; idx int32 [B,N,3] holds the
 * three nearest sources in ascending distance (ties: lower index first), weight fp32 [B,N,3]. */
EV2H_API int ev2h_three_nn_f32(const float *xyz1, int64_t q_stride_b, int64_t q_stride_c, int64_t q_stride_n,
                               const float *xyz2, int64_t s_stride_b, int64_t s_stride_c, int64_t s_stride_n,
                               int B, int N, int S, int32_t *idx, float *weight, ev2h_stream_t stream);
/* interpolated[b,n,:] = sum_k feats[b, idx[b,n,k], :] * weight[b,n,k]  (:301), written at column col
 * of out_rows [B*N, ld_out] (the concat with points1 happens by writing next to it).
 * feats_rows [B*S, ld_f], D channels.  Only columns col .. col + D - 1 of out_rows are written.  feats_rows and
 * out_rows need only the alignment of a float. */
EV2H_API int ev2h_three_interp_f32(const float *feats_rows, int ld_f, const int32_t *idx, const float *weight,
                                   int B, int N, int S, int D, float *out_rows, int ld_out, int col,
                                   ev2h_stream_t stream);

/* ---- event-window construction (SURVEY.md section 8f row N3) -------------------------------------
 * The step in front of the encoder: raw camera events -> the [5, N] point set (x, y, t, n_pos, n_neg).
 * Replaces the per-window numpy code of the reference's two dataset classes:
 *   EV2H_WINDOW_STREAM  ERPCParser.__getitem__, src/Ev2Hands/dataset/evaluation_stream.py:188-215
 *   EV2H_WINDOW_ERPC    Ev2HandSDataset.__getitem__, src/Ev2Hands/dataset/erpc.py:178-218 and :249
 * (np.add.at into 346x260 float32 grids, np.nonzero, mean time, [ERPC: * 1e-6, argsort by time, rebase,]
 * np.random.choice(M, N), pc_normalize).  Two calls, because the reference draws the N indices from numpy's
 * global generator with M, the number of occupied pixels, as the bound - the caller reads n_pixels back,
 * draws exactly like the reference, and passes the indices in (the same convention as the FPS start indices).
 *
 * events: float64 rows of row_stride doubles, columns 0..3 = x, y, t, polarity (any further columns are
 * ignored: the ERPC table carries two more); window b = rows [win_start[b], win_start[b] + win_count[b]),
 * win_count[b] <= max_count <= 16384 (STREAM) / 4096 (ERPC).  Every per-pixel sum is taken the way np.add.at
 * takes it: in double, rounded to the float32 cell, in stream order.  STREAM subtracts the window's first
 * timestamp from every t first (:188).  records: fp32 [B, max_count, 5] = (x, y, t_mean, n_pos, n_neg) of the
 * n_pixels[b] occupied pixels, in the reference's order right before the draw: np.nonzero (row-major) order
 * for STREAM, ascending mean time (pixel order among equal means, where the reference's unstable argsort may
 * return any order) with the earliest subtracted for ERPC.  Events outside the sensor are dropped and counted
 * in n_bad[b] (numpy would raise IndexError, or wrap negative indices). */
enum { EV2H_WINDOW_STREAM = 0, EV2H_WINDOW_ERPC = 1 };
EV2H_API int ev2h_window_aggregate_f64(const double *events, int64_t row_stride, const int64_t *win_start,
                                       const int32_t *win_count, int B, int max_count, int width, int height, int mode,
                                       float *records, int32_t *n_pixels, int32_t *n_bad, ev2h_stream_t stream);
/* out[b] = pc_normalize(records[b][sample_idx[b]]) transposed: fp32 [B, 5, N]; x -> 2 (x / width) - 1,
 * y -> 2 (y / height) - 1, t -> 2 ((t - t_min) / (t_max - t_min)) - 1 over the N drawn points (IEEE divisions in
 * the reference's operation order; a window whose drawn points share one time gives NaN like the reference).
 * sample_idx int64 [B, N], each in [0, n_pixels[b]); violations are counted into n_bad[b] (added to it). */
EV2H_API int ev2h_window_sample_f32(const float *records, int max_count, const int32_t *n_pixels, const int64_t *sample_idx,
                                    int B, int N, int width, int height, float *out, int32_t *n_bad, ev2h_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* EV2H_H */
