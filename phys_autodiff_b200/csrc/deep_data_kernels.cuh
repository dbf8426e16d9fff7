// Data-fit loss of deeper networks at caller-supplied points and its gradient with respect to every layer's weights:
//   L_d = (1/n_norm) sum_i sum_o lam[o] (y_io - target_io)^2,   y_i = MLP(x_i)
// for the network In = 4 -> H -> ... -> H -> Out = 4 set by physad_set_weights_deep (any L >= 1).  The term that anchors a
// physics-informed fit to initial conditions, boundary values or observations; it adds to the physics gradient of
// deep_grad_kernels.cuh / deep_tangent_kernels.cuh entry for entry.  ADDITIVE: no reference counterpart, checked against
// tests/deep_data_checker.c (itself pinned by finite differences and by oracle_mlp_forward_deep).
//
// Kernels (deep_data_kernels.cu; the source of k_deep_data_grad is deep_data_body.cuh):
//   k_deep_data_grad<H>   persistent, k_deep_grad's design with one row per point: forward with k_mlp_deep's arithmetic
//                         (bit-identical outputs to physad_mlp_forward_deep_dev), every layer's activations kept in a
//                         per-block checkpoint area, the output layer, seeds y_bar_o = coef_o (y_o - target_o) in fp32
//                         (coef_o = 2 lam_o / n_norm rounded to fp32; zero on tail rows), sum lam (y - target)^2 in double,
//                         then back-propagation through the output, hidden and first layers.  Weight gradients: fp32
//                         within a tile, then added into block-owned double partials (one owner per entry, no atomics).
//   k_deep_data_reduce    sums the block partials in block order (bitwise repeatable), writes grad[P] and the loss sum.
//
// Periodic-pair loss (deep_pair_kernels.cu): for B pairs of points (p_i, q_i),
//   L_p = (1/n_norm) sum_i sum_o lam[o] (y(p_i)_o - y(q_i)_o)^2,
// e.g. p on the face x_a = -1 and q = p + T_a e_a one period on, which states the periodic boundary condition of the grid
// calls' default domain at arbitrary points.  k_deep_pair_grad<H> is k_deep_data_grad's body run over the 2B rows of
// x[B][2] (row 2i = p_i, row 2i + 1 = q_i) with the partner row's outputs as the target: seeds
// y_bar(p_i) = coef (y(p_i) - y(q_i)) and y_bar(q_i) = -y_bar(p_i) exactly, the double sum counted once per pair; then
// k_deep_data_reduce.  The grid size, checkpoint area and partials are the data kernel's for 2B points.
// Vector-Jacobian product (vjp_points_kernels.cu): for caller-supplied cotangents y_bar[n][4],
//   grad = sum_i J_theta(y_i)^T y_bar_i,   the plain sum over the points (no scale: y_bar carries every weight),
// the gradient of any loss whose derivative with respect to y_i is y_bar_i.  k_vjp_points<H> is k_deep_data_grad's body
// with y_bar read from a.ybar (zero on tail rows) and no loss sum; then k_deep_data_reduce (acc[1] = 0).  With
// y_bar = coef (y - target) formed in fp32 it is k_deep_data_grad's gradient bit for bit.
// Gradient layout: that of physad_deep_loss_grad_dev (P = 9H + 4 + (L-1)(H^2 + H) doubles):
//   dW1 [H x 4] | db1 [H] | dWh [(L-1) x H x H, row-major [out][in]] | dbh [(L-1) x H] | dW2 [4 x H] | db2 [4]
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace physad {

struct DeepDataArgs {
    int hidden_layers;          // L >= 1
    long long n;                // points (> 0); pairs: rows, 2B
    const float4* x;            // [n] network inputs {x, y, z, t}; pairs: [B][2] (p_i, q_i)
    const float4* target;       // [n]; unused by the pair kernel
    const float* W1;            // [H][4] reference layout
    const float* b1;            // [H]
    const float* wh;            // [(L-1)][H][H] in k_mlp_deep's layout (input-major, output pairs stored (g+1, g))
    const float* bh;            // [(L-1)][H]
    const float* W2;            // [4][H] reference layout
    float coef[4];              // fp32(2 lam_o / n_norm): the seed scale
    double lam[4];              // loss weights of the double sum
    float* ckpt;                // [blocks][L][rows x H] activations of the current tile
    double* partials;           // [blocks][P + 1]
    // the VJP (vjp_points_launch), at the end so that no earlier field's offset moves; target, coef and lam are not read
    const float4* ybar;         // [n] cotangents of the outputs
};

constexpr int DEEP_DATA_THREADS = 256;

// Checkpoint floats one block needs for (H, L).
size_t deep_data_ckpt_floats(int H, int hidden_layers);
// Persistent grid size for n points (at most max_blocks).
int deep_data_blocks(int H, long long n_points, int max_blocks);
// k_deep_data_grad<H> on `blocks` blocks, then the block-order reduction into grad[P] and acc[1].  `mlp_const` points to a
// host MlpConst<H> (mlp_eval.cuh) whose w2 / b2 the output layer reads.  Returns a cudaError_t value.
int deep_data_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st);
// k_deep_pair_grad<H> on `blocks` blocks (a.n = 2B rows, a.target unused), then the same reduction.
int deep_pair_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st);
// k_vjp_points<H> on `blocks` blocks (a.ybar the seeds, a.target unused), then the same reduction (acc[1] = 0).
int vjp_points_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st);
// k_deep_data_reduce: partials [blocks][P + 1] summed in block order into grad[P] and acc[1].
int deep_data_reduce(const double* partials, int blocks, size_t P, double* grad, double* acc, cudaStream_t st);

}  // namespace physad
