// Closed loop for deeper networks: d(L_sigma + L_u) / d(every layer's weights) of the finite-difference physics loss,
// for the network In = 4 -> H -> ... -> H -> Out = 4 set by physad_set_weights_deep (L >= 2 hidden layers; L = 1 is the
// one-hidden-layer closed loop of grad_kernels.cuh).  ADDITIVE: no reference counterpart, checked against
// oracle_phys_loss_grad_deep (tests/deep_grad_checker.c, itself pinned by finite differences).
//
// Inputs are what the forward pass and k_phys_adjoint left in HBM: the four residual arrays (for A_+ = g / (2 dt)) and
// the time-t output adjoint A_t of every processed point.  Two kernels (deep_grad_kernels.cu):
//   k_deep_grad<H>        persistent, row-tiled like k_mlp_deep (a row = one (point, time slice) pair).  Per tile it
//                         recomputes the hidden layers in k_mlp_deep's exact operation order (so the ReLU masks are
//                         those of the fields that produced R), keeps every layer's activations of the tile in a
//                         per-block checkpoint area in global memory, then back-propagates
//                         y_bar = A_t | +A_+ | -A_+  (slices t, t+dt, t-dt) through the output, hidden and first layers.
//                         Weight gradients: fp32 within a tile, then added into block-owned double partials.
//   k_deep_grad_reduce    sums the block partials in block order (bitwise repeatable), writes grad[P] and the two
//                         residual sums.
// Gradient layout (P(H, L) = 9H + 4 + (L-1)(H^2 + H) doubles, the argument order of physad_set_weights_deep):
//   dW1 [H x 4] | db1 [H] | dWh [(L-1) x H x H, row-major [out][in]] | dbh [(L-1) x H] | dW2 [4 x H] | db2 [4]
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace physad {

struct DeepGradArgs {
    int nx, ny, nz;
    int z_begin, z_end;         // planes whose points are processed
    int z_origin;               // global z of plane 0 of the residual arrays
    int hidden_layers;          // L >= 2
    const float* cxs; const float* cys; const float* czs;   // axis coordinate tables (global indices)
    const float* W1;            // [H][4] reference layout
    const float* b1;            // [H]
    float tc[3];                // network time input of the slices t-dt, t, t+dt
    const float* wh;            // [(L-1)][H][H] in k_mlp_deep's layout (input-major, output pairs stored (g+1, g))
    const float* bh;            // [(L-1)][H]
    const float* W2;            // [4][H] reference layout
    const float* R[4];          // residuals, plane layout of the window starting at z_origin
    const float4* adj;          // A_t of the processed points (k_phys_adjoint)
    float scale_s, scale_u;     // 2 w / float(N) of the whole grid
    float inv2dt;               // 1 / (2 grid.dt) in fp32
    float* ckpt;                // [blocks][L][rows x H] activations of the current tile
    double* partials;           // [blocks][P + 2]
};

constexpr int DEEP_GRAD_THREADS = 256;

// Gradient length P(H, L) (0 for shapes that are not built).
size_t deep_grad_len(int H, int hidden_layers);
// Checkpoint floats one block needs for (H, L).
size_t deep_grad_ckpt_floats(int H, int hidden_layers);
// Persistent grid size for a slab of n_points points (at most max_blocks).
int deep_grad_blocks(int H, long long n_points, int max_blocks);
// k_deep_grad<H> on `blocks` blocks, then the block-order reduction into grad[P] and (if acc_out) the two sums.
// Returns a cudaError_t value.
int deep_grad_launch(int H, const DeepGradArgs& a, int blocks, double* grad, double* acc_out, cudaStream_t st);

}  // namespace physad
