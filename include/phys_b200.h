// Additive C++ entry points of the B200 build, in the style of include/phys.h / mlp_grid.h: the
// operations the reference planned but never shipped (SURVEY.md section 0 fact 2).  Host-pointer,
// void-returning, abort-with-message on CUDA errors, like the wrappers of the existing names.
#ifndef PHYS_AUTODIFF_PHYS_B200_H
#define PHYS_AUTODIFF_PHYS_B200_H

#include "mlp_grid.h"
#include "phys.h"

namespace phys {

// Loss forward on the single-kernel stencil with on-device reduction -- the
// cuda_phys_loss_forward_fused named in the reference's docs/PLAN_FUSED_PHYS_LOSS.md:59.
void cuda_phys_loss_forward_fused(const GridSpec& g, const PhysWeights& w, const float* sigma_tm1, const float* sigma_t,
                                  const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                                  float* out_loss_sigma, float* out_loss_u, float* opt_R_sigma = nullptr,
                                  float* opt_R_ux = nullptr, float* opt_R_uy = nullptr, float* opt_R_uz = nullptr);

// The whole hot path in one kernel: MLP at (x,y,z,t-dt|t|t+dt) over the grid -> residuals -> loss.
// Equivalent to mlp_generate_fields_cuda followed by cuda_phys_loss_forward_*, without any field
// ever leaving the chip (the "MLP -> physics mega-kernel" of docs/BENCHMARK_REPORT.md:61).
// Requires cfg.dims.In == cfg.dims.Out == 4 (what the reference's grid driver assumes, src/mlp_grid.cpp:69-80).  H <= 128 runs
// the fused kernel; wider networks run stage-wise (generic operator per slice, then the stencil + on-device reduction).
void mlp_phys_loss_fused_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw,
                              float t, float dt, float* out_loss_sigma, float* out_loss_u, float* opt_R_sigma = nullptr,
                              float* opt_R_ux = nullptr, float* opt_R_uy = nullptr, float* opt_R_uz = nullptr);

// The same PDE loss with the derivatives PROPAGATED THROUGH the MLP in forward mode instead of finite differences
// (BASELINE north-star's literal wording).  Additive and not the reference's arithmetic: the reference differences MLP
// outputs on the grid (src/phys_cpu.cpp:71-93), so the two losses differ by the discretisation error.  In = Out = 4, H <= 128.
void mlp_phys_loss_tangent_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw, float t,
                                float* out_loss_sigma, float* out_loss_u);

// Deeper networks (BASELINE config 5's depth sweep; additive -- the reference API has exactly one hidden layer,
// include/mlp.h:5-6): 4 -> H -> ... -> H -> 4 with hidden_layers >= 1 layers of width H in {32, 64, 128}, every layer the
// reference's layer rule (src/mlp_cpu.cpp:19-24).  Wh: (hidden_layers - 1) matrices [H x H] row-major [out][in]; bh:
// (hidden_layers - 1) x H.  tensor_cores = false: strict fp32, bit-identical to the CPU restatement of the rule;
// true: hidden -> hidden layers on tcgen05 with three-term bf16 operands (~1e-6 of the strict outputs, not bit-exact).
struct DeepMLPWeights {
    int hidden_layers = 1;
    std::vector<float> W1, b1, Wh, bh, W2, b2;
};
void mlp_phys_loss_deep_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw, float t,
                             float dt, float* out_loss_sigma, float* out_loss_u, bool tensor_cores = false);

// The closed loop the reference plans in REQUIREMENT.md:155-169 ("MLP backward: pass dL/dsigma, dL/du to the MLP
// weights") and stops short of (cpu_phys_loss_backward returns dL/dR only): the two losses of the MLP-generated
// fields AND d(L_sigma + L_u)/d(weights), the loss VJP carried through the transposed stencil and the MLP on the
// device.  `grad` is resized to the shapes of `w` (W1 [H x In], b1, W2 [Out x H], b2).  Same requirements as above.
void mlp_phys_loss_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw,
                             float t, float dt, float* out_loss_sigma, float* out_loss_u, MLPWeights& grad);

// The closed loop of the analytic loss: the two losses of mlp_phys_loss_tangent_cuda AND d(L_sigma + L_u)/d(weights), reverse
// mode over its forward-mode tangents in one kernel.  `grad` is resized to the shapes of `w`.  Same requirements as above.
void mlp_phys_loss_tangent_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw,
                                     float t, float* out_loss_sigma, float* out_loss_u, MLPWeights& grad);

// The closed loop of deeper networks: the two losses of mlp_phys_loss_deep_cuda (strict fp32) AND d(L_sigma + L_u) with
// respect to every layer's weights.  `grad` is resized to the shapes of `w` (grad.hidden_layers = w.hidden_layers).
void mlp_phys_loss_deep_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                  float t, float dt, float* out_loss_sigma, float* out_loss_u, DeepMLPWeights& grad);

// The analytic loss of a deep network: the derivatives of mlp_phys_loss_tangent_cuda propagated in forward mode through every
// layer of the DeepMLPWeights network (value row in the strict fp32 order of the deep forward, tangent rows with FMA), and its
// closed loop, d(L_sigma + L_u) with respect to every layer's weights.  `grad` is resized to the shapes of `w`.
void mlp_phys_loss_deep_tangent_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                     float t, float* out_loss_sigma, float* out_loss_u);
void mlp_phys_loss_deep_tangent_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w,
                                          const PhysWeights& pw, float t, float* out_loss_sigma, float* out_loss_u,
                                          DeepMLPWeights& grad);

// A deep network at arbitrary points: coords holds N inputs (x, y, z, t), already normalised like mlp_infer_cuda's; out is
// resized to N*4, AoS per point.  Strict fp32 in the arithmetic of the grid kernels (bit-identical to them at grid
// coordinates and to mlp_infer_cuda for hidden_layers = 1).  Every vector of `w` is checked against cfg and hidden_layers.
void mlp_infer_deep_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const std::vector<float>& coords, std::vector<float>& out);

// Data-fit loss of a deep network and its gradient with respect to every layer's weights: x and target hold B points of 4
// floats, lam 4 non-negative output weights or nullptr for 1/4 each (the mean((y - target)^2) of mlp_backward);
// *out_loss = (1/B) sum_i sum_o lam[o] (y_io - target_io)^2.  `grad` is resized to the shapes of `w` and adds directly to
// the physics gradient of mlp_phys_loss_deep_grad_cuda / mlp_phys_loss_deep_tangent_grad_cuda.  B = 0 gives zeros.
void mlp_data_loss_deep_grad_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, const float* target,
                                  std::size_t B, const float* lam, float* out_loss, DeepMLPWeights& grad);

// Periodic-pair loss of a deep network and its gradient with respect to every layer's weights: x holds B host pairs of two
// points of 4 floats, (p_i, q_i) (e.g. p on a face and q = p + T_a e_a one period on, T_a = f n_a / (n_a - 1)); lam as in
// mlp_data_loss_deep_grad_cuda; *out_loss = (1/B) sum_i sum_o lam[o] (y(p_i)_o - y(q_i)_o)^2.  `grad` is resized to the
// shapes of `w` and adds directly to mlp_data_loss_deep_grad_cuda's.  B = 0 gives zeros.  Every vector of `w` is checked
// against cfg.
void mlp_pair_loss_deep_grad_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, std::size_t B,
                                  const float* lam, float* out_loss, DeepMLPWeights& grad);

// The Jacobian of a deep network at arbitrary points: x holds B host points of 4 floats (network inputs, already
// normalised); y[B][4] gets the outputs (mlp_infer_deep_cuda's bit for bit) and J[B][4][4] the derivatives
// J[i][o][k] = dy_o / dc_k, formed exactly by forward-mode tangent rows.  B = 0 writes nothing.
void mlp_jacobian_deep_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, std::size_t B, float* y,
                            float* J);

// Derivative-fit loss of a deep network and its gradient with respect to every layer's weights (Neumann boundaries at
// points): x, dir and target hold B host rows of 4 floats; D_io = sum_k dir[i][k] J[i][o][k] and
// *out_loss = (1/B) sum_i sum_o lam[o] (D_io - target[i][o])^2 (lam as in mlp_data_loss_deep_grad_cuda).  For a zero
// normal derivative along space axis a, dir = dcdx[a] e_a and target = 0.  `grad` is resized to the shapes of `w` and
// adds directly to the data, pair and physics gradients; its b2 part is exactly zero.  B = 0 gives zeros.
void mlp_deriv_loss_deep_grad_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, const float* dir,
                                   const float* target, std::size_t B, const float* lam, float* out_loss, DeepMLPWeights& grad);

// Vector-Jacobian products of a deep network at arbitrary points: the gradient with respect to every layer's weights of any
// loss whose derivatives with respect to the outputs and the Jacobian are given.  x and ybar hold B host rows of 4 floats,
// Jbar B host blocks of 4 x 4 in mlp_jacobian_deep_cuda's J layout (Jbar[i][o][k] pairs with dy_o / dc_k).
// grad = sum_i ybar_i . dy_i/dtheta (+ sum_i Jbar_i : dJ_i/dtheta), the plain sum over the points with no scale; it adds
// directly to the other deep gradients.  `grad` is resized to the shapes of `w`.  B = 0 gives zeros.
void mlp_vjp_deep_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, const float* ybar, std::size_t B,
                       DeepMLPWeights& grad);
void mlp_jacobian_vjp_deep_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, const float* ybar,
                                const float* Jbar, std::size_t B, DeepMLPWeights& grad);

// The analytic loss of a deep network at arbitrary space-time points (collocation points) instead of the grid at one time:
// x holds B host points of 4 floats (x, y, z, t), the network inputs already normalised (the fourth is the grid's time input:
// t for MinusOneToOne, t + 0.5 for ZeroToOne); dcdx the 3 dc/dx of the space inputs (physad_grid_input_scales gives the
// grid's).  *out_loss_* = (w / B) sum R^2; opt_R, if given, receives B x 4 residuals {R_sigma, R_ux, R_uy, R_uz} per point.
// The _grad form also returns d(L_sigma + L_u) with respect to every layer's weights; `grad` is resized to the shapes of `w`
// and adds directly to mlp_data_loss_deep_grad_cuda's.  B = 0 gives zeros.  Every vector of `w` is checked against cfg.
void mlp_phys_loss_deep_tangent_points_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                            const float* x, std::size_t B, const float dcdx[3], float* out_loss_sigma,
                                            float* out_loss_u, float* opt_R = nullptr);
void mlp_phys_loss_deep_tangent_points_grad_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                                 const float* x, std::size_t B, const float dcdx[3], float* out_loss_sigma,
                                                 float* out_loss_u, DeepMLPWeights& grad);

}  // namespace phys

#endif  // PHYS_AUTODIFF_PHYS_B200_H
