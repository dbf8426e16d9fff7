// Data-fit loss of deeper networks at caller-supplied points and its gradient with respect to every layer's weights:
//   L_d = (1/n_norm) sum_i sum_o lam[o] (y_io - target_io)^2,   y_i = MLP(x_i)
// for the network In = 4 -> H -> ... -> H -> Out = 4 set by physad_set_weights_deep (any L >= 1).  The term that anchors a
// physics-informed fit to initial conditions, boundary values or observations; it adds to the physics gradient of
// deep_grad_kernels.cuh / deep_tangent_kernels.cuh entry for entry.  ADDITIVE: no reference counterpart, checked against
// tests/deep_data_checker.c (itself pinned by finite differences and by oracle_mlp_forward_deep).
//
// Two kernels (deep_data_kernels.cu):
//   k_deep_data_grad<H>   persistent, k_deep_grad's design with one row per point: forward with k_mlp_deep's arithmetic
//                         (bit-identical outputs to physad_mlp_forward_deep_dev), every layer's activations kept in a
//                         per-block checkpoint area, the output layer, seeds y_bar_o = coef_o (y_o - target_o) in fp32
//                         (coef_o = 2 lam_o / n_norm rounded to fp32; zero on tail rows), sum lam (y - target)^2 in double,
//                         then back-propagation through the output, hidden and first layers.  Weight gradients: fp32
//                         within a tile, then added into block-owned double partials (one owner per entry, no atomics).
//   k_deep_data_reduce    sums the block partials in block order (bitwise repeatable), writes grad[P] and the loss sum.
// Gradient layout: that of physad_deep_loss_grad_dev (P = 9H + 4 + (L-1)(H^2 + H) doubles):
//   dW1 [H x 4] | db1 [H] | dWh [(L-1) x H x H, row-major [out][in]] | dbh [(L-1) x H] | dW2 [4 x H] | db2 [4]
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace physad {

struct DeepDataArgs {
    int hidden_layers;          // L >= 1
    long long n;                // points (> 0)
    const float4* x;            // [n] network inputs {x, y, z, t}
    const float4* target;       // [n]
    const float* W1;            // [H][4] reference layout
    const float* b1;            // [H]
    const float* wh;            // [(L-1)][H][H] in k_mlp_deep's layout (input-major, output pairs stored (g+1, g))
    const float* bh;            // [(L-1)][H]
    const float* W2;            // [4][H] reference layout
    float coef[4];              // fp32(2 lam_o / n_norm): the seed scale
    double lam[4];              // loss weights of the double sum
    float* ckpt;                // [blocks][L][rows x H] activations of the current tile
    double* partials;           // [blocks][P + 1]
};

constexpr int DEEP_DATA_THREADS = 256;

// Checkpoint floats one block needs for (H, L).
size_t deep_data_ckpt_floats(int H, int hidden_layers);
// Persistent grid size for n points (at most max_blocks).
int deep_data_blocks(int H, long long n_points, int max_blocks);
// k_deep_data_grad<H> on `blocks` blocks, then the block-order reduction into grad[P] and acc[1].  `mlp_const` points to a
// host MlpConst<H> (mlp_eval.cuh) whose w2 / b2 the output layer reads.  Returns a cudaError_t value.
int deep_data_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st);

}  // namespace physad
