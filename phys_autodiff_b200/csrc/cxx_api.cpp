// The reference's C++ operator API (include/backend.h, mlp.h, mlp_grid.h, phys.h) implemented on
// the C-ABI of this library.  Same symbols, same host-pointer / void-return contract as the
// reference's src/mlp_cuda.cu, src/mlp_grid.cpp (the *_cuda half), src/phys_cuda_nonfused.cu and
// src/phys_cuda_fused.cu, so a caller links this library instead of those objects and nothing
// else changes.  Differences in behaviour, all deliberate:
//   * one lazily created, process-wide context keeps device scratch and weights alive between
//     calls (the reference cudaMalloc/cudaFree's everything per call, e.g. src/mlp_cuda.cu:94-120);
//   * every CUDA status is checked; a failure prints the message and aborts (the reference ignores
//     them, SURVEY.md section 5) -- still no exception crosses the boundary;
//   * the loss reduction runs on the device.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <random>

#include "../../include/phys_b200.h"
#include "../../include/physad_b200.h"

namespace {

std::mutex g_mu;  // the reference API is single-threaded; serialise rather than race on the shared context
physad_ctx* g_ctx = nullptr;

void die(const char* what, int rc) {
    std::fprintf(stderr, "phys_autodiff_b200: %s failed (%d, %s): %s\n", what, rc, physad_error_string(rc),
                 physad_last_error());
    std::abort();
}

physad_ctx* ctx() {
    if (!g_ctx) {
        if (int rc = physad_ctx_create(&g_ctx, -1)) die("physad_ctx_create", rc);
        std::atexit([] { physad_ctx_destroy(g_ctx); g_ctx = nullptr; });
    }
    return g_ctx;
}

physad_grid to_c(const phys::GridSpec& g) { return physad_grid{g.nx, g.ny, g.nz, g.hx, g.hy, g.hz, g.dt, g.periodic ? 1 : 0}; }
physad_phys_weights to_c(const phys::PhysWeights& w) { return physad_phys_weights{w.w_sigma, w.w_u}; }

void use_weights(physad_ctx* c, std::size_t In, std::size_t H, std::size_t Out, int norm, const float* W1, const float* b1,
                 const float* W2, const float* b2) {
    const physad_mlp_config cfg{int(In), int(H), int(Out), norm};
    if (int rc = physad_set_weights(c, &cfg, W1, b1, W2, b2)) die("physad_set_weights", rc);
}

int norm_of(phys::CoordNorm n) { return n == phys::CoordNorm::MinusOneToOne ? 1 : 0; }

}  // namespace

// ---- include/mlp.h ---------------------------------------------------------------------------
template <>
void mlp_forward<ExecCuda>(const float* x, const float* W1, const float* b1, const float* W2, const float* b2, float* y,
                           std::size_t B, std::size_t In, std::size_t H, std::size_t Out) {
    std::lock_guard<std::mutex> lk(g_mu);
    physad_ctx* c = ctx();
    use_weights(c, In, H, Out, 1, W1, b1, W2, b2);
    if (int rc = physad_mlp_forward_host(c, x, y, B)) die("mlp_forward<ExecCuda>", rc);
}

template <>
void mlp_backward<ExecCuda>(const float* x, const float* y_target, const float* W1, const float* b1, const float* W2,
                            const float* b2, float* dW1, float* db1, float* dW2, float* db2, std::size_t B,
                            std::size_t In, std::size_t H, std::size_t Out) {
    std::lock_guard<std::mutex> lk(g_mu);
    physad_ctx* c = ctx();
    use_weights(c, In, H, Out, 1, W1, b1, W2, b2);
    if (int rc = physad_mlp_backward_host(c, x, y_target, dW1, db1, dW2, db2, B)) die("mlp_backward<ExecCuda>", rc);
}

namespace phys {

// ---- include/mlp_grid.h ------------------------------------------------------------------------
// The stream of std::uniform_real_distribution is standard-library specific (reference
// src/mlp_grid.cpp:8-19 uses the same two std facilities), so this is the reference's generator by
// construction when built with the same libstdc++.
void mlp_random_init(MLPWeights& w, const MLPDims& d, std::uint32_t seed, float scale) {
    std::mt19937 gen(seed);
    std::uniform_real_distribution<float> dist(-scale, scale);
    auto fill = [&](std::vector<float>& v, std::size_t n) {
        v.resize(n);
        for (float& e : v) e = dist(gen);
    };
    fill(w.W1, d.H * d.In);
    fill(w.b1, d.H);
    fill(w.W2, d.Out * d.H);
    fill(w.b2, d.Out);
}

void make_grid_coords(const GridSpec& g, float t, CoordNorm norm, std::vector<float>& coords) {
    const bool m1p1 = norm == CoordNorm::MinusOneToOne;
    auto axis = [m1p1](int i, int n) {
        if (n <= 1) return 0.0f;
        const float u = float(i) / float(n - 1);
        return m1p1 ? 2.f * u - 1.f : u;
    };
    const float tt = m1p1 ? t : t + 0.5f;
    coords.resize(std::size_t(g.nx) * g.ny * g.nz * 4);
    float* p = coords.data();
    for (int z = 0; z < g.nz; ++z) {
        const float cz = axis(z, g.nz);
        for (int y = 0; y < g.ny; ++y) {
            const float cy = axis(y, g.ny);
            for (int x = 0; x < g.nx; ++x, p += 4) {
                p[0] = axis(x, g.nx); p[1] = cy; p[2] = cz; p[3] = tt;
            }
        }
    }
}

void mlp_infer_cuda(const MLPDims& d, const MLPWeights& w, const float* coords, std::size_t N, float* out) {
    mlp_forward<ExecCuda>(coords, w.W1.data(), w.b1.data(), w.W2.data(), w.b2.data(), out, N, d.In, d.H, d.Out);
}

void mlp_grid_infer_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, float t, std::vector<float>& out) {
    const std::size_t N = std::size_t(g.nx) * g.ny * g.nz;
    out.resize(N * cfg.dims.Out);
    if (cfg.dims.In == 4 && cfg.dims.Out == 4 && cfg.dims.H <= 128) {
        std::lock_guard<std::mutex> lk(g_mu);
        physad_ctx* c = ctx();
        use_weights(c, 4, cfg.dims.H, 4, norm_of(cfg.norm), w.W1.data(), w.b1.data(), w.W2.data(), w.b2.data());
        const physad_grid cg = to_c(g);
        if (int rc = physad_mlp_grid_infer_host(c, &cg, t, out.data())) die("mlp_grid_infer_cuda", rc);
        return;
    }
    // other shapes: explicit coordinate array through the generic operator, as the reference does
    std::vector<float> coords;
    make_grid_coords(g, t, cfg.norm, coords);
    mlp_infer_cuda(cfg.dims, w, coords.data(), N, out.data());
}

// Widths the grid kernels are not instantiated for (H > 128): the reference's own composition (src/mlp_grid.cpp:82-106) --
// explicit coordinates, the generic operator per time slice, split on the host -- so that the drop-in accepts every
// H the reference accepts.  In = Out = 4 is what the reference's grid driver itself assumes (its split hard-codes the
// stride 4, src/mlp_grid.cpp:69-80); other dims are rejected by the C-ABI with PHYSAD_E_UNSUPPORTED.
static bool grid_kernels_cover(const MLPGridConfig& cfg) { return cfg.dims.In != 4 || cfg.dims.Out != 4 || cfg.dims.H <= 128; }

static void generate_fields_generic(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, float t, float dt,
                                    std::vector<float>* sig[3], std::vector<float>* vel[3]) {
    const std::size_t N = std::size_t(g.nx) * g.ny * g.nz;
    const float ts[3] = {t - dt, t, t + dt};   // src/mlp_grid.cpp:87-89
    std::vector<float> coords, y(N * 4);
    for (int s = 0; s < 3; ++s) {
        make_grid_coords(g, ts[s], cfg.norm, coords);
        mlp_infer_cuda(cfg.dims, w, coords.data(), N, y.data());
        sig[s]->resize(N);
        vel[s]->resize(3 * N);
        float *ps = sig[s]->data(), *pu = vel[s]->data();
        for (std::size_t i = 0; i < N; ++i) {   // split_outputs_to_fields, src/mlp_grid.cpp:69-80
            ps[i] = y[i * 4];
            pu[i] = y[i * 4 + 1];
            pu[N + i] = y[i * 4 + 2];
            pu[2 * N + i] = y[i * 4 + 3];
        }
    }
}

void mlp_generate_fields_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, float t, float dt,
                              std::vector<float>& sigma_tm1, std::vector<float>& sigma_t, std::vector<float>& sigma_tp1,
                              std::vector<float>& u_tm1, std::vector<float>& u_t, std::vector<float>& u_tp1) {
    const std::size_t N = std::size_t(g.nx) * g.ny * g.nz;
    if (!grid_kernels_cover(cfg)) {
        std::vector<float>* sig[3] = {&sigma_tm1, &sigma_t, &sigma_tp1};
        std::vector<float>* vel[3] = {&u_tm1, &u_t, &u_tp1};
        generate_fields_generic(g, cfg, w, t, dt, sig, vel);
        return;
    }
    for (auto* s : {&sigma_tm1, &sigma_t, &sigma_tp1}) s->resize(N);
    for (auto* u : {&u_tm1, &u_t, &u_tp1}) u->resize(3 * N);
    std::lock_guard<std::mutex> lk(g_mu);
    physad_ctx* c = ctx();
    use_weights(c, cfg.dims.In, cfg.dims.H, cfg.dims.Out, norm_of(cfg.norm), w.W1.data(), w.b1.data(), w.W2.data(),
                w.b2.data());
    const physad_grid cg = to_c(g);
    if (int rc = physad_mlp_generate_fields_host(c, &cg, t, dt, sigma_tm1.data(), sigma_t.data(), sigma_tp1.data(),
                                                 u_tm1.data(), u_t.data(), u_tp1.data()))
        die("mlp_generate_fields_cuda", rc);
}

// ---- include/phys.h ----------------------------------------------------------------------------
#define PHYS_FIELDS sigma_tm1, sigma_t, sigma_tp1, u_tm1, u_t, u_tp1

void cuda_phys_residuals_fused_timed(const GridSpec& g, const float* sigma_tm1, const float* sigma_t,
                                     const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                                     float* R_sigma, float* R_ux, float* R_uy, float* R_uz, float* kernel_ms) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    if (int rc = physad_phys_residuals_host(ctx(), &cg, PHYS_FIELDS, R_sigma, R_ux, R_uy, R_uz, kernel_ms))
        die("cuda_phys_residuals", rc);
}

void cuda_phys_residuals_fused(const GridSpec& g, const float* sigma_tm1, const float* sigma_t, const float* sigma_tp1,
                               const float* u_tm1, const float* u_t, const float* u_tp1, float* R_sigma, float* R_ux,
                               float* R_uy, float* R_uz) {
    cuda_phys_residuals_fused_timed(g, PHYS_FIELDS, R_sigma, R_ux, R_uy, R_uz, nullptr);
}

void cuda_phys_residuals_nonfused_timed(const GridSpec& g, const float* sigma_tm1, const float* sigma_t,
                                        const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                                        float* R_sigma, float* R_ux, float* R_uy, float* R_uz, float* kernel_ms) {
    cuda_phys_residuals_fused_timed(g, PHYS_FIELDS, R_sigma, R_ux, R_uy, R_uz, kernel_ms);
}

void cuda_phys_residuals_nonfused(const GridSpec& g, const float* sigma_tm1, const float* sigma_t, const float* sigma_tp1,
                                  const float* u_tm1, const float* u_t, const float* u_tp1, float* R_sigma, float* R_ux,
                                  float* R_uy, float* R_uz) {
    cuda_phys_residuals_fused_timed(g, PHYS_FIELDS, R_sigma, R_ux, R_uy, R_uz, nullptr);
}

void cuda_phys_loss_forward_fused(const GridSpec& g, const PhysWeights& w, const float* sigma_tm1, const float* sigma_t,
                                  const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                                  float* out_loss_sigma, float* out_loss_u, float* opt_R_sigma, float* opt_R_ux,
                                  float* opt_R_uy, float* opt_R_uz) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(w);
    if (int rc = physad_phys_loss_host(ctx(), &cg, &cw, PHYS_FIELDS, out_loss_sigma, out_loss_u, opt_R_sigma, opt_R_ux,
                                       opt_R_uy, opt_R_uz))
        die("cuda_phys_loss_forward", rc);
}

void cuda_phys_loss_forward_nonfused(const GridSpec& g, const PhysWeights& w, const float* sigma_tm1, const float* sigma_t,
                                     const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                                     float* out_loss_sigma, float* out_loss_u, float* opt_R_sigma, float* opt_R_ux,
                                     float* opt_R_uy, float* opt_R_uz) {
    cuda_phys_loss_forward_fused(g, w, PHYS_FIELDS, out_loss_sigma, out_loss_u, opt_R_sigma, opt_R_ux, opt_R_uy, opt_R_uz);
}

void cuda_phys_loss_backward_nonfused(const GridSpec& g, const PhysWeights& w, const float* R_sigma, const float* R_ux,
                                      const float* R_uy, const float* R_uz, float* g_sigma, float* g_ux, float* g_uy,
                                      float* g_uz) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(w);
    if (int rc = physad_phys_backward_host(ctx(), &cg, &cw, R_sigma, R_ux, R_uy, R_uz, g_sigma, g_ux, g_uy, g_uz))
        die("cuda_phys_loss_backward_nonfused", rc);
}

void cuda_phys_loss_backward_fused(const GridSpec& g, const PhysWeights& w, const float* sigma_tm1, const float* sigma_t,
                                   const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                                   float* g_sigma, float* g_ux, float* g_uy, float* g_uz) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(w);
    if (int rc = physad_phys_backward_from_fields_host(ctx(), &cg, &cw, PHYS_FIELDS, g_sigma, g_ux, g_uy, g_uz))
        die("cuda_phys_loss_backward_fused", rc);
}
#undef PHYS_FIELDS

// ---- include/phys_b200.h --------------------------------------------------------------------------
void mlp_phys_loss_fused_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw,
                              float t, float dt, float* out_loss_sigma, float* out_loss_u, float* opt_R_sigma,
                              float* opt_R_ux, float* opt_R_uy, float* opt_R_uz) {
    if (!grid_kernels_cover(cfg)) {   // H > 128: stage-wise (fields through the generic operator, then the stencil + reduction)
        std::vector<float> s[3], u[3];
        std::vector<float>* sig[3] = {&s[0], &s[1], &s[2]};
        std::vector<float>* vel[3] = {&u[0], &u[1], &u[2]};
        generate_fields_generic(g, cfg, w, t, dt, sig, vel);
        cuda_phys_loss_forward_fused(g, pw, s[0].data(), s[1].data(), s[2].data(), u[0].data(), u[1].data(), u[2].data(),
                                     out_loss_sigma, out_loss_u, opt_R_sigma, opt_R_ux, opt_R_uy, opt_R_uz);
        return;
    }
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    if (int rc = physad_fused_loss_host(ctx(), &cg, &mc, w.W1.data(), w.b1.data(), w.W2.data(), w.b2.data(), &cw, t, dt,
                                        out_loss_sigma, out_loss_u, opt_R_sigma, opt_R_ux, opt_R_uy, opt_R_uz))
        die("mlp_phys_loss_fused_cuda", rc);
}

void mlp_phys_loss_tangent_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw, float t,
                                float* out_loss_sigma, float* out_loss_u) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    if (int rc = physad_tangent_loss_host(ctx(), &cg, &mc, w.W1.data(), w.b1.data(), w.W2.data(), w.b2.data(), &cw, t,
                                          out_loss_sigma, out_loss_u))
        die("mlp_phys_loss_tangent_cuda", rc);
}

void mlp_phys_loss_deep_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw, float t,
                             float dt, float* out_loss_sigma, float* out_loss_u, bool tensor_cores) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    physad_ctx* c = ctx();
    int rc = physad_set_weights_deep(c, &mc, w.hidden_layers, w.W1.data(), w.b1.data(), w.Wh.empty() ? nullptr : w.Wh.data(),
                                     w.bh.empty() ? nullptr : w.bh.data(), w.W2.data(), w.b2.data());
    if (!rc) rc = physad_set_deep_mode(c, tensor_cores ? 1 : 0);
    if (!rc) rc = physad_deep_loss_host(c, &cg, &cw, t, dt, out_loss_sigma, out_loss_u);
    physad_set_deep_mode(c, 0);
    if (rc) die("mlp_phys_loss_deep_cuda", rc);
}

void mlp_phys_loss_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw,
                             float t, float dt, float* out_loss_sigma, float* out_loss_u, MLPWeights& grad) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    grad.W1.resize(w.W1.size());
    grad.b1.resize(w.b1.size());
    grad.W2.resize(w.W2.size());
    grad.b2.resize(w.b2.size());
    if (int rc = physad_fused_loss_grad_host(ctx(), &cg, &mc, w.W1.data(), w.b1.data(), w.W2.data(), w.b2.data(), &cw, t, dt,
                                             out_loss_sigma, out_loss_u, grad.W1.data(), grad.b1.data(), grad.W2.data(),
                                             grad.b2.data()))
        die("mlp_phys_loss_grad_cuda", rc);
}

void mlp_phys_loss_tangent_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const MLPWeights& w, const PhysWeights& pw,
                                     float t, float* out_loss_sigma, float* out_loss_u, MLPWeights& grad) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    grad.W1.resize(w.W1.size());
    grad.b1.resize(w.b1.size());
    grad.W2.resize(w.W2.size());
    grad.b2.resize(w.b2.size());
    if (int rc = physad_tangent_loss_grad_host(ctx(), &cg, &mc, w.W1.data(), w.b1.data(), w.W2.data(), w.b2.data(), &cw, t,
                                               out_loss_sigma, out_loss_u, grad.W1.data(), grad.b1.data(), grad.W2.data(),
                                               grad.b2.data()))
        die("mlp_phys_loss_tangent_grad_cuda", rc);
}

void mlp_phys_loss_deep_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                  float t, float dt, float* out_loss_sigma, float* out_loss_u, DeepMLPWeights& grad) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    physad_ctx* c = ctx();
    grad.hidden_layers = w.hidden_layers;
    grad.W1.resize(w.W1.size());
    grad.b1.resize(w.b1.size());
    grad.Wh.resize(w.Wh.size());
    grad.bh.resize(w.bh.size());
    grad.W2.resize(w.W2.size());
    grad.b2.resize(w.b2.size());
    int rc = physad_set_weights_deep(c, &mc, w.hidden_layers, w.W1.data(), w.b1.data(), w.Wh.empty() ? nullptr : w.Wh.data(),
                                     w.bh.empty() ? nullptr : w.bh.data(), w.W2.data(), w.b2.data());
    if (!rc) rc = physad_deep_loss_grad_host(c, &cg, &cw, t, dt, out_loss_sigma, out_loss_u, grad.W1.data(), grad.b1.data(),
                                             grad.Wh.empty() ? nullptr : grad.Wh.data(), grad.bh.empty() ? nullptr : grad.bh.data(),
                                             grad.W2.data(), grad.b2.data());
    if (rc) die("mlp_phys_loss_deep_grad_cuda", rc);
}

namespace {
int set_deep(physad_ctx* c, const MLPGridConfig& cfg, const DeepMLPWeights& w) {
    const physad_mlp_config mc{int(cfg.dims.In), int(cfg.dims.H), int(cfg.dims.Out), norm_of(cfg.norm)};
    return physad_set_weights_deep(c, &mc, w.hidden_layers, w.W1.data(), w.b1.data(), w.Wh.empty() ? nullptr : w.Wh.data(),
                                   w.bh.empty() ? nullptr : w.bh.data(), w.W2.data(), w.b2.data());
}
}  // namespace

void mlp_phys_loss_deep_tangent_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                     float t, float* out_loss_sigma, float* out_loss_u) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    physad_ctx* c = ctx();
    static double* d_acc = nullptr;   // the two device sums; lives as long as the process's context
    int rc = set_deep(c, cfg, w);
    if (!rc && !d_acc) rc = int(cudaMalloc(&d_acc, 2 * sizeof(double)));
    if (!rc) rc = physad_deep_tangent_loss_dev(c, &cg, nullptr, t, d_acc, nullptr, nullptr, nullptr, nullptr, nullptr);
    double h_acc[2] = {0.0, 0.0};
    if (!rc) rc = int(cudaMemcpy(h_acc, d_acc, sizeof(h_acc), cudaMemcpyDeviceToHost));
    if (rc) die("mlp_phys_loss_deep_tangent_cuda", rc);
    physad_finalize_loss(h_acc, &cw, size_t(g.nx) * g.ny * g.nz, out_loss_sigma, out_loss_u);
}

void mlp_phys_loss_deep_tangent_grad_cuda(const GridSpec& g, const MLPGridConfig& cfg, const DeepMLPWeights& w,
                                          const PhysWeights& pw, float t, float* out_loss_sigma, float* out_loss_u,
                                          DeepMLPWeights& grad) {
    std::lock_guard<std::mutex> lk(g_mu);
    const physad_grid cg = to_c(g);
    const physad_phys_weights cw = to_c(pw);
    physad_ctx* c = ctx();
    grad.hidden_layers = w.hidden_layers;
    grad.W1.resize(w.W1.size());
    grad.b1.resize(w.b1.size());
    grad.Wh.resize(w.Wh.size());
    grad.bh.resize(w.bh.size());
    grad.W2.resize(w.W2.size());
    grad.b2.resize(w.b2.size());
    int rc = set_deep(c, cfg, w);
    if (!rc) rc = physad_deep_tangent_loss_grad_host(c, &cg, &cw, t, out_loss_sigma, out_loss_u, grad.W1.data(), grad.b1.data(),
                                                     grad.Wh.empty() ? nullptr : grad.Wh.data(),
                                                     grad.bh.empty() ? nullptr : grad.bh.data(), grad.W2.data(), grad.b2.data());
    if (rc) die("mlp_phys_loss_deep_tangent_grad_cuda", rc);
}

namespace {
// Every vector of a DeepMLPWeights against cfg and hidden_layers, before any pointer reaches the C-ABI (which reads
// exactly these sizes): a mismatch aborts with the offending field instead of reading past a vector.
void check_deep_shapes(const MLPGridConfig& cfg, const DeepMLPWeights& w, const char* what) {
    const std::size_t In = cfg.dims.In, H = cfg.dims.H, Out = cfg.dims.Out;
    const char* bad = nullptr;
    if (In != 4 || Out != 4 || (H != 32 && H != 64 && H != 128)) bad = "cfg.dims (In = Out = 4, H in {32, 64, 128})";
    else if (w.hidden_layers < 1 || w.hidden_layers > 16) bad = "hidden_layers (1 .. 16)";
    else {
        const std::size_t nl = std::size_t(w.hidden_layers - 1);
        if (w.W1.size() != H * In) bad = "W1.size() != H * In";
        else if (w.b1.size() != H) bad = "b1.size() != H";
        else if (w.Wh.size() != nl * H * H) bad = "Wh.size() != (hidden_layers - 1) * H * H";
        else if (w.bh.size() != nl * H) bad = "bh.size() != (hidden_layers - 1) * H";
        else if (w.W2.size() != Out * H) bad = "W2.size() != Out * H";
        else if (w.b2.size() != Out) bad = "b2.size() != Out";
    }
    if (bad) {
        std::fprintf(stderr, "phys_autodiff_b200: %s: %s\n", what, bad);
        std::abort();
    }
}
}  // namespace

void mlp_infer_deep_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const std::vector<float>& coords, std::vector<float>& out) {
    std::lock_guard<std::mutex> lk(g_mu);
    check_deep_shapes(cfg, w, "mlp_infer_deep_cuda");
    if (coords.size() % 4) {
        std::fprintf(stderr, "phys_autodiff_b200: mlp_infer_deep_cuda: coords.size() is not a multiple of 4\n");
        std::abort();
    }
    const std::size_t N = coords.size() / 4;
    out.resize(N * 4);
    physad_ctx* c = ctx();
    int rc = set_deep(c, cfg, w);
    if (!rc) rc = physad_mlp_forward_deep_host(c, coords.data(), out.data(), N);
    if (rc) die("mlp_infer_deep_cuda", rc);
}

void mlp_data_loss_deep_grad_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const float* x, const float* target,
                                  std::size_t B, const float* lam, float* out_loss, DeepMLPWeights& grad) {
    std::lock_guard<std::mutex> lk(g_mu);
    check_deep_shapes(cfg, w, "mlp_data_loss_deep_grad_cuda");
    physad_ctx* c = ctx();
    grad.hidden_layers = w.hidden_layers;
    grad.W1.resize(w.W1.size());
    grad.b1.resize(w.b1.size());
    grad.Wh.resize(w.Wh.size());
    grad.bh.resize(w.bh.size());
    grad.W2.resize(w.W2.size());
    grad.b2.resize(w.b2.size());
    int rc = set_deep(c, cfg, w);
    if (!rc) rc = physad_deep_data_loss_grad_host(c, x, target, B, lam, out_loss, grad.W1.data(), grad.b1.data(),
                                                  grad.Wh.empty() ? nullptr : grad.Wh.data(),
                                                  grad.bh.empty() ? nullptr : grad.bh.data(), grad.W2.data(), grad.b2.data());
    if (rc) die("mlp_data_loss_deep_grad_cuda", rc);
}

void mlp_phys_loss_deep_tangent_points_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                            const float* x, std::size_t B, const float dcdx[3], float* out_loss_sigma,
                                            float* out_loss_u, float* opt_R) {
    std::lock_guard<std::mutex> lk(g_mu);
    check_deep_shapes(cfg, w, "mlp_phys_loss_deep_tangent_points_cuda");
    const physad_phys_weights cw = to_c(pw);
    physad_ctx* c = ctx();
    const std::size_t bytes = B * 4 * sizeof(float);
    float *d_x = nullptr, *d_R = nullptr;
    double* d_acc = nullptr;
    double h_acc[2] = {0.0, 0.0};
    int rc = set_deep(c, cfg, w);
    if (!rc) rc = int(cudaMalloc(&d_acc, 2 * sizeof(double)));
    if (!rc && B) rc = int(cudaMalloc(&d_x, bytes));
    if (!rc && B && opt_R) rc = int(cudaMalloc(&d_R, bytes));
    if (!rc && B) rc = int(cudaMemcpy(d_x, x, bytes, cudaMemcpyHostToDevice));
    if (!rc) rc = physad_deep_tangent_points_loss_dev(c, d_x, B, dcdx, d_acc, d_R, nullptr);
    if (!rc) rc = int(cudaMemcpy(h_acc, d_acc, sizeof(h_acc), cudaMemcpyDeviceToHost));
    if (!rc && d_R) rc = int(cudaMemcpy(opt_R, d_R, bytes, cudaMemcpyDeviceToHost));
    cudaFree(d_x);
    cudaFree(d_R);
    cudaFree(d_acc);
    if (rc) die("mlp_phys_loss_deep_tangent_points_cuda", rc);
    physad_finalize_loss(h_acc, &cw, B ? B : 1, out_loss_sigma, out_loss_u);
}

void mlp_phys_loss_deep_tangent_points_grad_cuda(const MLPGridConfig& cfg, const DeepMLPWeights& w, const PhysWeights& pw,
                                                 const float* x, std::size_t B, const float dcdx[3], float* out_loss_sigma,
                                                 float* out_loss_u, DeepMLPWeights& grad) {
    std::lock_guard<std::mutex> lk(g_mu);
    check_deep_shapes(cfg, w, "mlp_phys_loss_deep_tangent_points_grad_cuda");
    const physad_phys_weights cw = to_c(pw);
    physad_ctx* c = ctx();
    grad.hidden_layers = w.hidden_layers;
    grad.W1.resize(w.W1.size());
    grad.b1.resize(w.b1.size());
    grad.Wh.resize(w.Wh.size());
    grad.bh.resize(w.bh.size());
    grad.W2.resize(w.W2.size());
    grad.b2.resize(w.b2.size());
    int rc = set_deep(c, cfg, w);
    if (!rc) rc = physad_deep_tangent_points_loss_grad_host(c, x, B, dcdx, &cw, out_loss_sigma, out_loss_u, grad.W1.data(),
                                                            grad.b1.data(), grad.Wh.empty() ? nullptr : grad.Wh.data(),
                                                            grad.bh.empty() ? nullptr : grad.bh.data(), grad.W2.data(),
                                                            grad.b2.data());
    if (rc) die("mlp_phys_loss_deep_tangent_points_grad_cuda", rc);
}

}  // namespace phys

// C-ABI access to the weight generator for non-C++ hosts (bench.py, tests): see include/physad_b200.h.
extern "C" void physad_mlp_random_init(int In, int H, int Out, unsigned int seed, float scale, float* W1, float* b1,
                                       float* W2, float* b2) {
    phys::MLPWeights w;
    phys::MLPDims d;
    d.In = std::size_t(In); d.H = std::size_t(H); d.Out = std::size_t(Out);
    phys::mlp_random_init(w, d, seed, scale);
    std::copy(w.W1.begin(), w.W1.end(), W1);
    std::copy(w.b1.begin(), w.b1.end(), b1);
    std::copy(w.W2.begin(), w.W2.end(), W2);
    std::copy(w.b2.begin(), w.b2.end(), b2);
}
