/*
 * d3h_lbs.h -- C ABI of the skinning stage behind the extraction (SURVEY.md section 8(f) row 4).
 *
 * D3-Human moves every extracted vertex from the canonical pose to the frame's pose with linear-blend skinning
 * (geometry/hmsdf.py:471, 508, 582, 618 -> deform/smplx_exavatar_deformer.py:434-486):
 *     interpolate_weights :363-383   nearest SMPL-X template vertex of every point (pytorch3d knn_points, K = self.k = 1,
 *                                    :39), its skinning weights
 *     apply_lbs_inverse   :385-421   per POINT: M_p = sum_j w[p,j] A_j (P x J x 16 multiply-adds), torch.inverse of P 4x4
 *                                    matrices, one 4x4 product -- twice per call (:474-476)
 * on all Va rows of verts_aug, although >= 80 % of them are the zeroed, unreferenced boundary slots (gshell_tets.py:423-
 * 427).  With K = 1 the blended matrix depends on the point only through its nearest template vertex, so everything per
 * point collapses to per TEMPLATE VERTEX tables (10 475 rows instead of ~230 000), and the zero rows share one result:
 *     B[v] = sum_j lbs_weights[v,j] A_j;   posed[p] = B_pose[nn(p)] (B_init[nn(p)]^-1 [p;1]) + trans
 *
 * Conventions as in d3h_tets.h: raw device pointers, row-major fp32, 4x4 matrices as 16 consecutive floats, 0 / negative
 * D3H_E_* return codes with d3h_last_error_string(), caller-owned memory, everything enqueued on `stream`.
 */
#ifndef D3H_LBS_H_
#define D3H_LBS_H_

#include <stdint.h>

#include "d3h_tets.h"

#ifdef __cplusplus
extern "C" {
#endif

/* B[v] = sum_j lbs_weights[v,j] A[j]  (lbs_weights (Vt,J), A (J,16), out (Vt,16)); invert != 0 stores B[v]^-1 instead
 * (Gauss-Jordan with partial pivoting per template vertex; the reference inverts per point, :413). */
int d3h_lbs_blend(const float* lbs_weights, const float* a, int64_t n_template, int32_t n_joints, int32_t invert, float* out,
                  d3h_stream_t stream);

/* Nearest template vertex of every point (knn_points with K = 1: smallest squared distance, lowest index on ties).
 * Compaction-aware: the rows of `pts` that are exactly (0,0,0) -- the unreferenced rows of verts_aug -- are not searched
 * one by one, they all take the result of ONE search for the origin.  idx (P) int32.
 * workspace: d3h_lbs_nearest_workspace_bytes(P) bytes, 16-byte aligned. */
int64_t d3h_lbs_nearest_workspace_bytes(int64_t n_points);
int d3h_lbs_nearest(const float* pts, int64_t n_points, const float* tmpl, int64_t n_template, int32_t* idx, void* workspace,
                    int64_t workspace_bytes, d3h_stream_t stream);

/* posed[p] = (B_pose[idx[p]] [can;1])[:3] + trans,  can = (B_init_inv[idx[p]] [pts[p];1])[:3]   (:474-476)
 * b_pose == NULL: only the canonical points are produced (lbs_forward_inverse, :424-430) and `posed` may be NULL.
 * canonical (P,3) is an output either way (the backward pass reads it).  trans (3) may be NULL. */
int d3h_lbs_apply(const float* pts, int64_t n_points, const int32_t* idx, const float* b_init_inv, const float* b_pose,
                  const float* trans, float* canonical, float* posed, d3h_stream_t stream);

/* Adjoint of d3h_lbs_apply for an upstream gradient g_posed (P,3):
 *   g_pts[p]   = (B_pose[idx] B_init_inv[idx])[:3,:3]^T g_posed[p]            (overwritten)
 *   g_b[v]    += sum over the points with idx[p] = v of g_posed[p] (x) [can[p];1]   (Vt,12: the first three rows of B_pose)
 *   g_trans   += sum_p g_posed[p]                                              (3), may be NULL
 * g_b / g_trans ACCUMULATE (zero them first).  `pts` (the forward input, may be NULL) lets the kernel sum the upstream
 * gradients of the all-zero rows per CTA instead of through twelve atomics per row on one table row.  The zero rows need
 * not share one idx: per CTA the zero rows of one idx are summed, the others take the per-row atomics.  The result is the
 * same as with pts == NULL up to the order of the float additions. */
int d3h_lbs_apply_backward(const float* g_posed, int64_t n_points, const int32_t* idx, const float* b_init_inv,
                           const float* b_pose, const float* canonical, const float* pts, float* g_pts, float* g_b,
                           float* g_trans, d3h_stream_t stream);

/* g_a[j] (16 floats, last row zero) = sum_v lbs_weights[v,j] g_b[v]   (overwritten) */
int d3h_lbs_blend_backward(const float* lbs_weights, const float* g_b, int64_t n_template, int32_t n_joints, float* g_a,
                           d3h_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* D3H_LBS_H_ */
