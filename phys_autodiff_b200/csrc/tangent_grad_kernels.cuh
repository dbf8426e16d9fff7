// Gradient of the analytic ("tangent") physics loss with respect to the MLP weights: reverse mode over the forward-mode
// loss of tangent_kernels.cuh, so that the loss physad_tangent_loss_dev reports can be trained on.  Additive (no
// reference counterpart); checked against an fp32-faithful restatement that central differences pin (tests/test_tangent_grad.py).
//
// Per point, with c = (cx, cy, cz, ct), z_h = b1_h + W1[h,:] c, m_h = [z_h > 0], a_h = m_h z_h, y = b2 + W2 a,
// J[o][k] = sum_h m_h W2[o,h] W1[h,k], g[o][j] = s_j J[o][j], div = g[1][0] + g[2][1] + g[3][2]:
//   R_o = J[o][3] + sum_j y_{j+1} g[o][j],   R_0 += y_0 div
// and with gb_o = (2 w_o / float(N)) R_o (fp32, as the finite-difference closed loop):
//   yb_0 = gb_0 div,   yb_{j+1} = sum_o gb_o g[o][j],   Jb[o][3] = gb_o,   Jb[o][j] = s_j (gb_o y_{j+1} + [o = j+1] gb_0 y_0)
// The mask is piecewise constant, so with dz_h = m_h sum_o W2[o,h] yb_o and S_h[o][k] = sum_points m_h Jb[o][k]:
//   db2_o = sum yb_o                     dW2[o,h] = sum yb_o a_h + sum_k W1[h,k] S_h[o][k]
//   db1_h = sum dz_h                     dW1[h,k] = sum dz_h c_k + sum_o W2[o,h] S_h[o][k]     (k = 3: c_t sum dz_h + ...)
// The 16 masked sums S_h are shared by dW1 and dW2 and contracted with the weights once, by the last block.
//
// k_tangent_grad (tangent_grad_kernels.cu): persistent blocks of 256 threads over chunks of 256 points, two phases a chunk.
//   stage     thread per point: the tangent forward with k_tangent_loss's roundings in the same order (scalar fma.rn gives
//             the bits of one lane of its fma.rn.f32x2), the two residual square sums in double, c | yb | Jb to shared memory;
//   backward  thread per (hidden unit, group of HT points): z_h recomputed in the forward's strict order (the same masks),
//             24 accumulators per unit (S_h 16 | sum yb a 4 | sum dz c 3 | sum dz 1), fp32 over 32 points, double beyond.
// Block partials, summed in block order by the last block to finish (bitwise repeatable), then the contraction into the
// reference layouts  dW1[H*4] | db1[H] | dW2[4*H] | db2[4]  (runtime H).  No FFMA2 (packed fused multiply-adds are kept to
// the kernels tests/test_boundary.py names): the masked sums use predicated FADD2, everything else scalar FFMA.
#pragma once
#include <cuda_runtime.h>

namespace physad {

struct TangentGradArgs {
    int nx, ny, nz, z_begin, z_end;
    const float* cxs; const float* cys; const float* czs;   // axis coordinate tables (global indices)
    float sx, sy, sz;          // dc/dx of the three space coordinates
    float scale_s, scale_u;    // 2 w / float(N) of the whole grid
    float ct;                  // network time input
    const float *W1, *W2;      // device copies, reference layout (the last block's contraction)
    int H;                     // runtime width (<= template width)
    double* partials;          // [gridDim.x][TGRAD_NACC * HT + 6]
    unsigned int* ticket;
    double* acc;               // [2]: sum R_sigma^2, sum |R_u|^2 over the processed points
    double* grad;              // [9 H + 4]
};

constexpr int TGRAD_THREADS = 256;
constexpr int TGRAD_NACC = 24;

// tangent_const: host TangentConst<HT> (tangent_kernels.cuh) for HT in {32, 64, 128}; both return cudaError_t values
int tangent_grad_blocks_per_sm(int HT, int* out);
int tangent_grad_launch(int HT, const void* tangent_const, const TangentGradArgs& a, unsigned blocks, cudaStream_t st);

}  // namespace physad
