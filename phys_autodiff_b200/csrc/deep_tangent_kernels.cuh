// Analytic ("tangent") physics loss of deeper networks and its gradient with respect to every layer's weights, for the
// network In = 4 -> H -> ... -> H -> Out = 4 set by physad_set_weights_deep (on the grid L >= 2 hidden layers, L = 1 being
// physad_tangent_loss_* of tangent_kernels.cuh / tangent_grad_kernels.cuh; at points any L >= 1).  ADDITIVE: no reference
// counterpart, checked against tests/deep_tangent_checker.c (itself pinned by finite differences).
//
// Per point the network runs on 5 rows: the value row a and the four tangent rows a_dot_k = da/dc_k (k = x, y, z, t):
//   layer 1   z = b1 + W1 c                  k_mlp_deep's strict fp32 roundings and order (W1[h,3] t pre-rounded);
//             m = z > 0, a = relu(z), a_dot_k = m (.) W1[:,k]        (exact)
//   hidden l  z = bh_l + Wh_l a              strict: from the bias, inputs ascending, separate multiply and add
//             z_dot_k = Wh_l a_dot_k         scalar fma.rn from +0, inputs ascending
//             m = z > 0 (value row only), a = relu(z), a_dot_k = m (.) z_dot_k
//   output    y = b2 + W2 a (strict), J[:,k] = W2 a_dot_k (fma.rn from +0, h ascending)
// so the value path is bit-identical to k_mlp_deep at slice t.  The residuals are k_tangent_loss's:
//   d/dx_j = s_j J[:,j], d/dt = J[:,3];  R_sigma = d_t sigma + u . grad(sigma) + sigma div(u),  R_u = d_t u + (u . grad) u.
//
// Three kernels (deep_tangent_kernels.cu, colloc_tangent_kernels.cu; the body is deep_tangent_body.cuh):
//   k_deep_tangent<H, GRAD>  persistent, row-tiled like k_mlp_deep / k_deep_grad (a lane holds the 5 rows of one point).
//                            GRAD = false: forward, residuals (optional), the two double sums per block.
//                            GRAD = true:  the same forward with every layer's activations kept in a per-block checkpoint
//                            area, the output seeds of DESIGN section 4.6.1 formed in registers, then reverse mode through
//                            every layer.  Weight gradients in fp32 within a tile, then added to block-owned double partials.
//   k_colloc_tangent<H, GRAD>  the same at caller-supplied points (x, y, z, t) instead of the grid (collocation points):
//                            one float4 per point, its own time input; residuals (optional) AoS per point.
//   k_deriv_tangent<H, GRAD>  the points kernel with another last stage (deriv_tangent_kernels.cu): GRAD = false writes
//                            y and J per point; GRAD = true the derivative-fit loss of DESIGN section 4.13 and its gradient.
//   k_vjp_tangent<H, true>   the points kernel seeded with the caller's cotangents (vjp_tangent_kernels.cu):
//                            grad = sum_i (J_theta(y_i)^T y_bar_i + J_theta(J_i)^T : J_bar_i), the plain sum over the
//                            points; the output layer's values are not computed.
//   k_deep_tangent_reduce    sums the block partials in block order (bitwise repeatable): grad[P] and the two sums.
// Gradient layout: that of deep_grad_kernels.cuh,  dW1 | db1 | dWh | dbh | dW2 | db2  (P = 9H + 4 + (L-1)(H^2 + H)).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace physad {

struct DeepTangentArgs {
    int nx, ny, nz;
    int z_begin, z_end;         // planes whose points are processed
    int hidden_layers;          // L >= 2 (grid), >= 1 (points)
    const float* cxs; const float* cys; const float* czs;   // axis coordinate tables (global indices)
    const float* W1;            // [H][4] reference layout
    const float* b1;            // [H]
    float tc;                   // network time input at t
    const float* wh;            // [(L-1)][H][H] in k_mlp_deep's layout (input-major, output pairs stored (g+1, g))
    const float* bh;            // [(L-1)][H]
    const float* W2;            // [4][H] reference layout
    const float* b2;            // [4]
    float sx, sy, sz;           // dc/dx of the three space coordinates
    float scale_s, scale_u;     // 2 w / float(N) of the whole grid (GRAD only)
    float* R[4];                // slab-local residual outputs or null (loss only)
    float* ckpt;                // [blocks][L][rows x H] activations of the current tile (GRAD only)
    double* partials;           // [blocks][P + 2] (GRAD) or [blocks][2]
    // points mode (colloc_tangent_launch): the rows are n_points caller-supplied inputs {c_x, c_y, c_z, c_t}; nx .. tc,
    // z_begin, z_end and R are not read
    const float4* pts;
    long long n_points;
    float4* R_pts;              // [n_points] {R_sigma, R_ux, R_uy, R_uz} or null (loss only)
    // derivative mode (deriv_tangent_launch), at the end so that no earlier field's offset moves; sx .. scale_u and R_pts
    // are not read
    const float4* dirs;         // [n_points] direction d_i in network coordinates (GRAD)
    const float4* targets;      // [n_points] target g_i of the four directional derivatives (GRAD)
    float coef[4];              // float(2 lam_o / n_norm) (GRAD)
    double lam[4];              // lam_o of the un-normalised sum (GRAD)
    float4* y_pts;              // [n_points] outputs y (not GRAD)
    float4* J_pts;              // [n_points][4] rows J[o][0..3] = dy_o / dc_k (not GRAD)
    // VJP mode (vjp_tangent_launch), at the end likewise; sx .. scale_u, R_pts and the derivative fields are not read
    const float4* ybar;         // [n_points] cotangents of y
    const float4* Jbar;         // [n_points][4] cotangents of J, row o = {J_bar[o][0..3]} (the layout of J_pts)
};

constexpr int DEEP_TANGENT_THREADS = 256;

// Checkpoint floats one block needs for L hidden layers.
size_t deep_tangent_ckpt_floats(int hidden_layers);
// Persistent grid size for a slab of n_points points (at most max_blocks).
int deep_tangent_blocks(int H, long long n_points, int max_blocks);
// k_deep_tangent<H, grad> on `blocks` blocks, then the block-order reduction into acc[2] and (grad) grad[P].
// Returns a cudaError_t value.
int deep_tangent_launch(int H, bool grad, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st);
// The same kernel body with its rows taken from a.pts (one float4 load per point, W1[h,3] c_t rounded per row), as
// k_colloc_tangent<H, grad> (colloc_tangent_kernels.cu), then the same reduction: at the grid's own coordinates the
// sums, residuals and gradient equal deep_tangent_launch's bit for bit.  Any hidden_layers >= 1.
int colloc_tangent_launch(int H, bool grad, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st);
// The same body at a.pts as k_deriv_tangent<H, grad> (deriv_tangent_kernels.cu), any hidden_layers >= 1.  grad = false:
// the Jacobian query, y and J of every point into a.y_pts / a.J_pts, no partials and no reduction (acc and grad_out
// unused).  grad = true: the derivative-fit loss of DESIGN section 4.13 and its gradient, then deep_tangent_reduce, whose
// acc[2] is {sum_i sum_o lam_o (D_io - g_io)^2, 0}.
int deriv_tangent_launch(int H, bool grad, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st);
// The same body at a.pts as k_vjp_tangent<H, true> (vjp_tangent_kernels.cu), any hidden_layers >= 1: seeds a.ybar (value
// row) and a.Jbar (tangent rows), then deep_tangent_reduce, whose acc[2] is {0, 0}.
int vjp_tangent_launch(int H, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st);
// k_deep_tangent_reduce: the block partials [blocks][P + 2] summed in block order into grad[P] and acc[2].
int deep_tangent_reduce(const double* partials, int blocks, size_t P, double* acc, double* grad, cudaStream_t st);

}  // namespace physad
