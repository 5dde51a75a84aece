/*
 * d3h_mlp.h -- C ABI of the SDF field query that feeds the extraction (SURVEY.md section 8(f) row 3).
 *
 * D3-Human evaluates `self.sdf_net(v_deformed)` on ALL N grid vertices before every extraction
 * (geometry/hmsdf.py:434-444, 528-538): positional encoding (geometry/embedding.py:4-38, n_freq = 6 -> 39 channels)
 * followed by geometry/mlp.py:9-45 -- Linear(39,256), 6 x Linear(256,256) with the encoding concatenated again in front
 * of hidden layer 3 (skip_in = [3]: Linear(295,256)), Softplus(beta=100) after each, Linear(256,1) -- in fp32
 * (train.py:1622-1626).  That is 0.83 MFLOP per vertex, 1.8 TFLOP per forward pass at 128^3: the FLOP sink of an
 * iteration, and GEMM-shaped, so unlike the extraction it belongs on the tensor cores.
 *
 * The entry points below are the building blocks the Python host (d3human-code_b200/geometry/mlp.py, a drop-in for the
 * reference's `MLP` module with the same parameters / state_dict) chains for the forward and backward pass, and for the
 * second derivative the eikonal term needs (section "Second derivative" below).  The GEMMs run on the 5th-generation
 * tensor cores (tcgen05.mma kind::tf32, accumulators in tensor memory) with the 3xTF32 split
 *     a = a_hi + a_lo,  a_hi = a with the low 13 mantissa bits cleared:   a.b ~= a_hi.b_hi + a_lo.b_hi + a_hi.b_lo
 * so the results carry fp32-level error (~1e-6 relative, like a reordered fp32 sum) -- the reference computes in fp32
 * with TF32 disabled (torch default), and sign(sdf) decides the topology downstream.
 *
 * Conventions as in d3h_tets.h: raw device pointers, row-major fp32 with explicit leading dimensions (in floats), 0 /
 * negative D3H_E_* return codes with d3h_last_error_string(), caller-owned memory, everything enqueued on `stream`.
 */
#ifndef D3H_MLP_H_
#define D3H_MLP_H_

#include <stdint.h>

#include "d3h_tets.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Embedding.forward (geometry/embedding.py:23-38): out[m, 0:3] = x[m], then for k < n_freq:
 * out[m, 3+6k : 6+6k] = sin(2^k x[m]), out[m, 6+6k : 9+6k] = cos(2^k x[m]); columns [3(2 n_freq + 1), n_cols) are set
 * to zero (padding up to the GEMM's K granularity).  `out` has leading dimension ld >= n_cols. */
int d3h_mlp_embed(const float* x, int64_t m, int32_t n_freq, float* out, int64_t ld, int32_t n_cols,
                  d3h_stream_t stream);

/* Its adjoint: g_x[m] (+)= g_emb[m,0:3] + sum_k 2^k (cos(2^k x) g_sin_k - sin(2^k x) g_cos_k).  accumulate != 0 adds
 * to g_x, otherwise g_x is overwritten. */
int d3h_mlp_embed_backward(const float* x, int64_t m, int32_t n_freq, const float* g_emb, int64_t ld, float* g_x,
                           int32_t accumulate, d3h_stream_t stream);

/* The weight operand of d3h_mlp_linear in the layout the kernel consumes: B (n_pad x k_pad, zero outside the valid
 * part) split into hi / lo and stored as the shared-memory image of every 32-column slice, so that the kernel fetches a
 * slice with one bulk copy.  Run once per call and weight (the weights change every optimiser step; 8 n_pad k_pad bytes):
 *     B[n][k] = transpose ? w[(row0 + k) ldw + col0 + n] : w[(row0 + n) ldw + col0 + k]     for n < n_valid, k < k_valid
 * transpose = 0 packs nn.Linear.weight (rows = outputs) for the forward pass, transpose = 1 its transpose (or a column
 * slice of it) for the input gradient.  n_pad in {64, 128, 192, 256}, k_pad % 32 == 0, `packed` 16-byte aligned. */
int64_t d3h_mlp_packed_weight_bytes(int32_t n_pad, int32_t k_pad);
int d3h_mlp_pack_weight(const float* w, int64_t ldw, int32_t n_valid, int32_t k_valid, int32_t transpose, int32_t row0,
                        int32_t col0, int32_t n_pad, int32_t k_pad, float* packed, d3h_stream_t stream);

/* One nn.Linear (+ activation) of MLP.net on the tensor cores:
 *     c[m, n] = f( sum_k a[m, k] B[n, k] + bias[n] )
 *   a (M, lda), B = `w_packed` (d3h_mlp_pack_weight with n_pad = N, k_pad = K), c (M, ldc)
 *   K % 32 == 0 (zero-pad the input columns), N in {64, 128, 192, 256}, all pointers 16-byte aligned, lda / ldc / ldy
 *   multiples of 4.  bias may be NULL.
 *   mode 0: f = identity
 *   mode 1: f = Softplus(beta = 100, threshold = 20)                      (geometry/mlp.py:16,27)
 *   mode 2: c = (a B^T) * softplus'(z) with softplus'(z) = 1 - exp(-100 y) recovered from the layer's saved OUTPUT
 *           y = softplus(z) given in `y` (M, ldy) -- the backward pass through the activation of the previous layer. */
int d3h_mlp_linear(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                   const float* bias, int32_t mode, const float* y, int64_t ldy, float* c, int64_t ldc,
                   d3h_stream_t stream);

/* Weight / bias gradient of one nn.Linear: dw[n, k] += sum_m dz[m, n] a[m, k], db[n] += sum_m dz[m, n]
 * (dw, db ACCUMULATE: zero them first).  dz (M, ldz) with N in {128, 256}; a (M, lda) with K in {64, 128, 192, 256};
 * dw (N, lddw).  db may be NULL.  Tensor cores as above, contraction over the M points: every CTA owns a range of
 * points and writes its partial product to `workspace` (d3h_mlp_wgrad_workspace_bytes, 16-byte aligned), a second kernel
 * adds the partial products to dw / db. */
int64_t d3h_mlp_wgrad_workspace_bytes(int64_t m, int32_t n, int32_t k);
int d3h_mlp_wgrad(const float* dz, int64_t ldz, const float* a, int64_t lda, int64_t m, int32_t n, int32_t k, float* dw,
                  int64_t lddw, float* db, void* workspace, int64_t workspace_bytes, d3h_stream_t stream);

/* The output layer Linear(K, d_out) for small d_out (1 for the SDF): out[m, j] = sum_k a[m, k] w[j, k] + bias[j]. */
int d3h_mlp_head(const float* a, int64_t lda, int64_t m, int32_t k, const float* w, const float* bias, int32_t d_out,
                 float* out, d3h_stream_t stream);

/* Its backward pass in one sweep over a (the saved output of the last hidden layer, softplus applied):
 *   dz[m, k] = (sum_j g[m, j] w[j, k]) * (1 - exp(-100 a[m, k]))      gradient at the last hidden pre-activation
 *   dw[j, k] += sum_m g[m, j] a[m, k],  db[j] += sum_m g[m, j]        (ACCUMULATE)
 * K <= 256 and a multiple of 4, lda / ldz multiples of 4, a / dz / w 16-byte aligned. */
int d3h_mlp_head_backward(const float* a, int64_t lda, int64_t m, int32_t k, const float* w, int32_t d_out,
                          const float* g, float* dz, int64_t ldz, float* dw, float* db, d3h_stream_t stream);

/* ---- Second derivative (the eikonal term: autograd.grad(sdf, x, create_graph=True), then a loss on that gradient).
 * With delta_l the gradient at the pre-activation z_l of hidden layer l from the first backward pass, g_emb the gradient at
 * the encoding, and an upstream v (M, 3) for the first backward's g_x: a tangent pass along x' = v (e' = E'(x) v,
 * z'_l = h'_l W_l^T, a'_l = z'_l * softplus'(z_l)), then an adjoint pass from the output layer down
 *     mu_l      = (mu_{l+1} W_{l+1})[activation part] * softplus'(z_l) + beta [beta a_l <= 20] exp(-beta a_l) delta_l z'_l
 *     dW_l     += mu_l^T h_l + delta_l^T h'_l,  db_l += sum mu_l     (d3h_mlp_wgrad, two calls per input block)
 *     gbar     += (mu_l W_l)[encoding part]
 *     g_x       = E'(x)^T gbar + E''(x)[v]^T g_emb
 * with softplus'' recovered from the saved output a = softplus(z) as in mode 2 of d3h_mlp_linear and zero past the
 * threshold, as torch's softplus double backward. */

/* e' = E'(x) v: out[m, 0:3] = v[m], out[m, 3+6k+d] = 2^k cos(2^k x) v, out[m, 6+6k+d] = -2^k sin(2^k x) v; columns up to
 * n_cols are zeroed.  Layout rules as d3h_mlp_embed (x, v (M, 3) contiguous). */
int d3h_mlp_embed_tangent(const float* x, const float* v, int64_t m, int32_t n_freq, float* out, int64_t ld, int32_t n_cols,
                          d3h_stream_t stream);

/* g_x[m] = E'(x)^T gbar[m] + sum_k -4^k v (sin(2^k x) g_emb_sin_k + cos(2^k x) g_emb_cos_k), overwritten.  gbar may be NULL
 * (the standalone Embedding: only the second term). */
int d3h_mlp_embed_second_backward(const float* x, const float* v, int64_t m, int32_t n_freq, const float* gbar,
                                  int64_t ldbar, const float* g_emb, int64_t ld, float* g_x, d3h_stream_t stream);

/* Tangent through one hidden layer, same GEMM as d3h_mlp_linear (no bias): zdot = a B^T, adot = zdot * softplus'(z) with
 * softplus' from the layer's saved output y (M, ldy).  Rules of d3h_mlp_linear; y / zdot / adot hold N columns. */
int d3h_mlp_linear_tangent(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                           const float* y, int64_t ldy, float* zdot, int64_t ldzd, float* adot, int64_t ldad,
                           d3h_stream_t stream);

/* Adjoint step: c = (a B^T) * softplus'(z) + beta [beta y <= 20] exp(-beta y) * delta * zdot, where y, delta and zdot are
 * the saved output, first-backward gradient and tangent of the layer that produced the GEMM's output columns.  Rules of
 * d3h_mlp_linear; y / delta / zdot / c hold N columns. */
int d3h_mlp_linear_adjoint(const float* a, int64_t lda, int64_t m, int32_t k, const float* w_packed, int32_t n,
                           const float* y, int64_t ldy, const float* delta, int64_t ldd, const float* zdot, int64_t ldzd,
                           float* c, int64_t ldc, d3h_stream_t stream);

/* The output layer's share in one sweep: dw[j, k] += sum_m g[m, j] adot[m, k] (ACCUMULATE; the output bias gets no second
 * derivative) and mu[m, k] = beta [beta a <= 20] exp(-beta a) delta zdot for the last hidden layer (a, delta, zdot at m, k).
 * K <= 256 and a multiple of 4, leading dimensions multiples of 4, adot / a / delta / zdot / mu 16-byte aligned. */
int d3h_mlp_head_second_backward(const float* adot, int64_t ldad, const float* a, int64_t lda, const float* delta,
                                 int64_t ldd, const float* zdot, int64_t ldzd, int64_t m, int32_t k, const float* g,
                                 int32_t d_out, float* dw, float* mu, int64_t ldmu, d3h_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* D3H_MLP_H_ */
