/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the Jacobian of deeper networks at arbitrary points and the derivative-fit
 * loss with its gradient with respect to every layer's weights (tests/test_deep_deriv.py compiles it into a temporary
 * shared library, -ffp-contract=off):
 *   D_io = sum_k d_ik J[i][o][k],  acc = sum_i sum_o lam[o] (D_io - g_io)^2,  L_g = acc / n_norm,  grad = dL_g / d(weights)
 * for In = 4 -> H -> ... -> H -> Out = 4 with L >= 1 hidden layers, x, dir (d) and target (g) [B][4].
 * PARITY UNPINNED (no reference counterpart).  The per-point forward is that of deep_tangent_checker.c (included through
 * deep_tangent_points_checker.c): point_f, the kernel-faithful value row and tangent rows, and point_d, all in double.
 * The five-row adjoint is oracle_deep_tangent_points_loss_grad's, restated here with the derivative loss's seeds:
 * value row y_bar = 0, tangent row k J_bar[o][k] = coef_o e_o d_k.  Two modes:
 *   all_double = 0  kernel-faithful: point_f; D_o = ((d_x J[o][0] + d_y J[o][1]) + d_z J[o][2]) + d_t J[o][3] and
 *                   e_o = D_o - g_o in fp32, every operation rounded; coef_o = float(2 lam_o / n_norm), the seeds
 *                   (coef_o e_o) d_k in fp32; acc from double(D_o) - double(g_o); the adjoint in double.
 *   all_double = 1  everything in double: the function whose central finite differences pin the adjoint.
 * Parameters and gradient in the argument order of physad_set_weights_deep.  lam NULL: 1/4 each.
 */
#include "deep_tangent_points_checker.c"

/* y[B*4] and J[B*16] (J[i*16 + o*4 + k] = dy_o / dc_k) of the faithful forward: what the CUDA Jacobian call computes */
int oracle_jacobian_deep(int H, int L, const double* theta, const float* x, size_t B, float* y, float* J) {
    if (H < 1 || L < 1) return -1;
    const size_t NG = dt_len(H, L);
    float* th = (float*)malloc(sizeof(float) * NG);
    float* act = (float*)malloc(sizeof(float) * (size_t)L * NR * H);
    for (size_t e = 0; e < NG; ++e) th[e] = (float)theta[e];
    for (size_t i = 0; i < B; ++i) point_f(H, L, th, x + 4 * i, act, y + 4 * i, J + 16 * i);
    free(th); free(act);
    return 0;
}

int oracle_deriv_loss_grad_deep(int H, int L, const double* theta, const float* x, const float* dir, const float* target,
                                size_t B, const float* lam_in, size_t n_norm, int all_double, double* acc_out, double* grad) {
    if (H < 1 || L < 1 || n_norm == 0) return -1;
    const size_t NG = dt_len(H, L), nl = (size_t)(L - 1), HH = (size_t)H * H;
    float lam[4] = {0.25f, 0.25f, 0.25f, 0.25f};
    if (lam_in) memcpy(lam, lam_in, sizeof(lam));
    float* th_f = (float*)malloc(sizeof(float) * NG);
    for (size_t e = 0; e < NG; ++e) th_f[e] = (float)theta[e];
    const double* th = theta;
    const double *Wh = th + 5 * H, *W2 = th + 5 * H + nl * (HH + H);
    float* af = (float*)malloc(sizeof(float) * (size_t)L * NR * H);
    double* ad = (double*)malloc(sizeof(double) * (size_t)L * NR * H);
    double* da = (double*)malloc(sizeof(double) * NR * H);
    double* dp = (double*)malloc(sizeof(double) * NR * H);
    for (size_t e = 0; e < NG; ++e) grad[e] = 0.0;
    double *dW1 = grad, *db1 = grad + 4 * H, *dWh = grad + 5 * H, *dbh = dWh + nl * HH, *dW2 = dbh + nl * H, *db2 = dW2 + 4 * H;
    double acc = 0.0;
    for (size_t i = 0; i < B; ++i) {
        const float cf[4] = {x[i * 4], x[i * 4 + 1], x[i * 4 + 2], x[i * 4 + 3]};
        const double cd[4] = {cf[0], cf[1], cf[2], cf[3]};
        const float* d = dir + 4 * i;
        const float* g = target + 4 * i;
        double seed[NR][4];
        for (int o = 0; o < 4; ++o) seed[0][o] = 0.0;
        if (all_double) {
            double y[4], J[16];
            point_d(H, L, th, cd, ad, y, J);
            for (int o = 0; o < 4; ++o) {
                double D = 0.0;
                for (int k = 0; k < 4; ++k) D += (double)d[k] * J[o * 4 + k];
                const double e = D - (double)g[o];
                acc += (double)lam[o] * (e * e);
                for (int k = 0; k < 4; ++k) seed[1 + k][o] = 2.0 * (double)lam[o] / (double)n_norm * e * (double)d[k];
            }
        } else {
            float yf[4], Jf[16];
            point_f(H, L, th_f, cf, af, yf, Jf);
            for (size_t e = 0; e < (size_t)L * NR * H; ++e) ad[e] = af[e];
            for (int o = 0; o < 4; ++o) {
                const float D = ((d[0] * Jf[o * 4] + d[1] * Jf[o * 4 + 1]) + d[2] * Jf[o * 4 + 2]) + d[3] * Jf[o * 4 + 3];
                const float e = D - g[o];
                const double dd = (double)D - (double)g[o];
                acc += (double)lam[o] * (dd * dd);
                const float coef = (float)(2.0 * (double)lam[o] / (double)n_norm);
                const float ce = coef * e;
                for (int k = 0; k < 4; ++k) seed[1 + k][o] = (double)(ce * d[k]);
            }
        }
        /* output layer (the value-row seed is zero, so db2 stays +0) */
        const double* aL = ad + nl * NR * H;
        for (int o = 0; o < 4; ++o) db2[o] += seed[0][o];
        for (int r = 0; r < NR; ++r)
            for (int h = 0; h < H; ++h) {
                double v = 0.0;
                for (int o = 0; o < 4; ++o) {
                    dW2[o * H + h] += seed[r][o] * aL[(size_t)r * H + h];
                    v += W2[o * H + h] * seed[r][o];
                }
                da[(size_t)r * H + h] = v;
            }
        /* hidden layers, last to first: every row masked by the value row's mask */
        for (size_t l = nl; l >= 1; --l) {
            const double *a_out = ad + l * NR * H, *a_in = ad + (l - 1) * NR * H, *W = Wh + (l - 1) * HH;
            for (int gg = 0; gg < H; ++gg) {
                const int m = a_out[gg] > 0.0;
                for (int r = 0; r < NR; ++r) {
                    const double dv = m ? da[(size_t)r * H + gg] : 0.0;
                    da[(size_t)r * H + gg] = dv;
                    for (int h = 0; h < H; ++h) dWh[(l - 1) * HH + (size_t)gg * H + h] += dv * a_in[(size_t)r * H + h];
                }
                dbh[(l - 1) * H + gg] += da[gg];
            }
            for (int r = 0; r < NR; ++r)
                for (int h = 0; h < H; ++h) {
                    double v = 0.0;
                    for (int gg = 0; gg < H; ++gg) v += W[(size_t)gg * H + h] * da[(size_t)r * H + gg];
                    dp[(size_t)r * H + h] = v;
                }
            for (size_t e = 0; e < (size_t)NR * H; ++e) da[e] = dp[e];
        }
        /* layer 1: dW1[h,k] += delta_value c_k + delta_tan,k, db1 += delta_value */
        for (int h = 0; h < H; ++h) {
            if (!(ad[h] > 0.0)) continue;
            db1[h] += da[h];
            for (int k = 0; k < 4; ++k) dW1[h * 4 + k] += da[h] * cd[k] + da[(size_t)(1 + k) * H + h];
        }
    }
    *acc_out = acc;
    free(th_f); free(af); free(ad); free(da); free(dp);
    return 0;
}
