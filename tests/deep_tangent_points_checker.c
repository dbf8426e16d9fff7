/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the analytic loss of deeper networks at arbitrary points (collocation
 * points) and its gradient with respect to every layer's weights (tests/test_deep_tangent_points.py compiles it into a
 * temporary shared library, -ffp-contract=off).
 *
 * PARITY UNPINNED: the reference has no such function.  Per point the body of oracle_deep_tangent_loss_grad
 * (deep_tangent_checker.c, included below), with the point's inputs c = x[i] (x, y, z, t; already normalised) instead of
 * the grid's coordinates, the three space scales dcdx[] given instead of formed from the grid, and the mean over n_norm
 * instead of the grid's N:
 *   all_double = 0  kernel-faithful: point_f, R rounded to float, seeds (2.f * w / (float)n_norm) * (float)R in fp32;
 *   all_double = 1  everything in double (point_d), seeds 2 w / n_norm R: the function finite differences pin.
 * Outputs: the two sums (not normalised), R[B*4] = {R_sigma, R_ux, R_uy, R_uz} per point (optional) and the gradient of
 * L_sigma + L_u = (w_sigma / n_norm) sum R_sigma^2 + (w_u / n_norm) sum |R_u|^2 in the layout of deep_tangent_checker.c.
 */
#include "deep_tangent_checker.c"

int oracle_deep_tangent_points_loss_grad(int H, int L, const double* theta, size_t B, const float* x, const double dcdx[3],
                                         float w_sigma, float w_u, size_t n_norm, int all_double, double* acc_s,
                                         double* acc_u, float* Rout, double* grad) {
    if (L < 1 || n_norm == 0) return -1;
    const size_t NG = dt_len(H, L), nl = (size_t)(L - 1), HH = (size_t)H * H;
    float* th_f = (float*)malloc(sizeof(float) * NG);
    for (size_t i = 0; i < NG; ++i) th_f[i] = (float)theta[i];
    const double* th = theta;
    const double *Wh = th + 5 * H, *W2 = th + 5 * H + nl * (HH + H);
    float* af = (float*)malloc(sizeof(float) * (size_t)L * NR * H);
    double* ad = (double*)malloc(sizeof(double) * (size_t)L * NR * H);
    double* da = (double*)malloc(sizeof(double) * NR * H);
    double* dp = (double*)malloc(sizeof(double) * NR * H);
    if (grad)
        for (size_t i = 0; i < NG; ++i) grad[i] = 0.0;
    double *dW1 = grad, *db1 = grad ? grad + 4 * H : 0, *dWh = grad ? grad + 5 * H : 0, *dbh = grad ? dWh + nl * HH : 0;
    double *dW2 = grad ? dbh + nl * H : 0, *db2 = grad ? dW2 + 4 * H : 0;
    const double* s = dcdx;
    double as = 0.0, au = 0.0;
    for (size_t i = 0; i < B; ++i) {
        const float cf[4] = {x[i * 4], x[i * 4 + 1], x[i * 4 + 2], x[i * 4 + 3]};
        const double cd[4] = {cf[0], cf[1], cf[2], cf[3]};
        double y[4], J[4][4];
        if (all_double) {
            point_d(H, L, th, cd, ad, y, (double*)J);
        } else {
            float yf[4], Jf[16];
            point_f(H, L, th_f, cf, af, yf, Jf);
            for (size_t e = 0; e < (size_t)L * NR * H; ++e) ad[e] = af[e];
            for (int o = 0; o < 4; ++o) {
                y[o] = yf[o];
                for (int k = 0; k < 4; ++k) J[o][k] = Jf[o * 4 + k];
            }
        }
        double gr[4][3];
        for (int o = 0; o < 4; ++o)
            for (int j = 0; j < 3; ++j) gr[o][j] = J[o][j] * s[j];
        const double div = gr[1][0] + gr[2][1] + gr[3][2];
        double R[4];
        for (int o = 0; o < 4; ++o) R[o] = J[o][3] + (y[1] * gr[o][0] + y[2] * gr[o][1] + y[3] * gr[o][2]);
        R[0] += y[0] * div;
        if (!all_double)
            for (int o = 0; o < 4; ++o) R[o] = (double)(float)R[o];
        if (Rout)
            for (int o = 0; o < 4; ++o) Rout[i * 4 + o] = (float)R[o];
        as += R[0] * R[0];
        au += R[1] * R[1] + R[2] * R[2] + R[3] * R[3];
        if (!grad) continue;
        /* output seeds (DESIGN section 4.6.1) */
        double gb[4];
        for (int o = 0; o < 4; ++o) {
            const float w = o == 0 ? w_sigma : w_u;
            gb[o] = all_double ? 2.0 * (double)w / (double)n_norm * R[o] : (double)((2.f * w / (float)n_norm) * (float)R[o]);
        }
        double seed[NR][4];
        seed[0][0] = gb[0] * div;
        for (int j = 0; j < 3; ++j) seed[0][j + 1] = gb[0] * gr[0][j] + gb[1] * gr[1][j] + gb[2] * gr[2][j] + gb[3] * gr[3][j];
        for (int o = 0; o < 4; ++o) {
            seed[4][o] = gb[o];
            for (int j = 0; j < 3; ++j) seed[1 + j][o] = s[j] * (gb[o] * y[j + 1] + (o == j + 1 ? gb[0] * y[0] : 0.0));
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
                    const double d = m ? da[(size_t)r * H + gg] : 0.0;
                    da[(size_t)r * H + gg] = d;
                    for (int h = 0; h < H; ++h) dWh[(l - 1) * HH + (size_t)gg * H + h] += d * a_in[(size_t)r * H + h];
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
    *acc_s = as;
    *acc_u = au;
    free(th_f); free(af); free(ad); free(da); free(dp);
    return 0;
}
