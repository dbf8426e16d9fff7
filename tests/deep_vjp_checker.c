/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the vector-Jacobian products of deeper networks at arbitrary points
 * (tests/test_deep_vjp.py compiles it into a temporary shared library, -ffp-contract=off):
 *   grad = sum_i (sum_o ybar_io dy_io / dtheta + sum_o sum_k Jbar_iok dJ_iok / dtheta)
 * for In = 4 -> H -> ... -> H -> Out = 4 with L >= 1 hidden layers, x and ybar [B][4], Jbar [B][4][4] (Jbar[i][o][k] pairs
 * with J[i][o][k] = dy_o / dc_k) or NULL for zeros.  PARITY UNPINNED (no reference counterpart).
 * The per-point forward is that of deep_tangent_checker.c (point_f: the kernel-faithful value and tangent rows; point_d:
 * all in double).  The five-row adjoint is the one of oracle_deriv_loss_grad_deep (deep_deriv_checker.c) and of
 * oracle_deep_tangent_points_loss_grad, restated with the caller's seeds: value row ybar, tangent row k the column
 * Jbar[.][k].  With Jbar = 0 the tangent rows carry zeros and the adjoint is the one of oracle_data_loss_grad_deep
 * (deep_data_checker.c, included too) with its seeds given.  Two modes:
 *   all_double = 0  kernel-faithful activations (point_f), the adjoint in double;
 *   all_double = 1  everything in double: the gradient of oracle_vjp_objective, whose central finite differences pin it.
 * Parameters and gradient in the argument order of physad_set_weights_deep.
 */
#include "deep_deriv_checker.c"
#include "deep_data_checker.c"

/* sum_i (sum_o ybar_io y_io + sum_ok Jbar_iok J_iok) in double (point_d): the function whose gradient the VJP is */
int oracle_vjp_objective(int H, int L, const double* theta, const float* x, const float* ybar, const float* Jbar, size_t B,
                         double* out) {
    if (H < 1 || L < 1) return -1;
    double* ad = (double*)malloc(sizeof(double) * (size_t)L * NR * H);
    double s = 0.0;
    for (size_t i = 0; i < B; ++i) {
        const double cd[4] = {x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]};
        double y[4], J[16];
        point_d(H, L, theta, cd, ad, y, J);
        for (int o = 0; o < 4; ++o) s += (double)ybar[4 * i + o] * y[o];
        if (Jbar)
            for (int e = 0; e < 16; ++e) s += (double)Jbar[16 * i + e] * J[e];
    }
    *out = s;
    free(ad);
    return 0;
}

int oracle_jacobian_vjp_deep(int H, int L, const double* theta, const float* x, const float* ybar, const float* Jbar,
                             size_t B, int all_double, double* grad) {
    if (H < 1 || L < 1) return -1;
    const size_t NG = dt_len(H, L), nl = (size_t)(L - 1), HH = (size_t)H * H;
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
    for (size_t i = 0; i < B; ++i) {
        const float cf[4] = {x[i * 4], x[i * 4 + 1], x[i * 4 + 2], x[i * 4 + 3]};
        const double cd[4] = {cf[0], cf[1], cf[2], cf[3]};
        double seed[NR][4];
        for (int o = 0; o < 4; ++o) {
            seed[0][o] = (double)ybar[4 * i + o];
            for (int k = 0; k < 4; ++k) seed[1 + k][o] = Jbar ? (double)Jbar[16 * i + 4 * o + k] : 0.0;
        }
        if (all_double) {
            double y[4], J[16];
            point_d(H, L, th, cd, ad, y, J);
        } else {
            float yf[4], Jf[16];
            point_f(H, L, th_f, cf, af, yf, Jf);
            for (size_t e = 0; e < (size_t)L * NR * H; ++e) ad[e] = af[e];
        }
        /* output layer */
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
    free(th_f); free(af); free(ad); free(da); free(dp);
    return 0;
}

/* the value-only form: Jbar = 0 */
int oracle_vjp_deep(int H, int L, const double* theta, const float* x, const float* ybar, size_t B, int all_double,
                    double* grad) {
    return oracle_jacobian_vjp_deep(H, L, theta, x, ybar, NULL, B, all_double, grad);
}
