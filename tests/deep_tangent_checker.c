/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the analytic loss of deeper networks and its closed loop
 * (tests/test_deep_tangent.py compiles it into a temporary shared library): the forward-mode physics loss of
 * In = 4 -> H -> ... -> H -> Out = 4 with L >= 1 hidden layers and d(L_sigma + L_u) / d(every layer's weights).
 *
 * PARITY UNPINNED: the reference has no such function.  Per point the network runs on the value row a and the four
 * tangent rows a_dot_k = da/dc_k (k = x, y, z, t); residuals as oracle_tangent_loss (oracle/oracle.c).  Two modes:
 *   all_double = 0  kernel-faithful: the value row in strict fp32 (oracle_mlp_forward_deep's arithmetic), the tangent
 *                   rows with fmaf from +0 for inputs ascending, the order of k_deep_tangent; R formed in double from
 *                   the fp32 y and J and rounded to float; g = (2w/float(N)) R in fp32; the adjoint runs in double.
 *                   This is what the CUDA kernel is compared with (compile with -ffp-contract=off).
 *   all_double = 1  everything in double, masks from double pre-activations: the function whose central finite
 *                   differences pin the adjoint.
 * Parameters and gradient in the argument order of physad_set_weights_deep:
 *   W1[H*4] | b1[H] | Wh[(L-1)*H*H, row-major [out][in]] | bh[(L-1)*H] | W2[4*H] | b2[4]
 */
#include <math.h>

#include "../oracle/oracle_grad.c"

#define NR 5 /* rows per point: value, d/dc_x, d/dc_y, d/dc_z, d/dc_t */

static size_t dt_len(int H, int L) { return (size_t)9 * H + 4 + (size_t)(L - 1) * ((size_t)H * H + H); }

/* act[(l*NR + r)*H + h]: row r of hidden layer l+1 after the ReLU / mask; y[o], J[o*4 + k] = dy_o / dc_k. */
static void point_f(int H, int L, const float* th, const float c[4], float* act, float y[4], float J[16]) {
    const size_t nl = (size_t)(L - 1), HH = (size_t)H * H;
    const float *W1 = th, *b1 = th + 4 * H, *Wh = th + 5 * H, *bh = Wh + nl * HH, *W2 = bh + nl * H, *b2 = W2 + 4 * H;
    for (int h = 0; h < H; ++h) {
        float s = b1[h];
        for (int k = 0; k < 4; ++k) s += W1[h * 4 + k] * c[k];
        const int m = s > 0.f;
        act[h] = m ? s : 0.f;
        for (int k = 0; k < 4; ++k) act[(size_t)(1 + k) * H + h] = m ? W1[h * 4 + k] : 0.f;
    }
    for (size_t l = 0; l < nl; ++l) {
        const float *W = Wh + l * HH, *in = act + l * NR * H;
        float* out = act + (l + 1) * NR * H;
        for (int g = 0; g < H; ++g) {
            float s = bh[l * H + g], tk[4] = {0.f, 0.f, 0.f, 0.f};
            for (int h = 0; h < H; ++h) s += W[(size_t)g * H + h] * in[h];
            for (int k = 0; k < 4; ++k)
                for (int h = 0; h < H; ++h) tk[k] = fmaf(W[(size_t)g * H + h], in[(size_t)(1 + k) * H + h], tk[k]);
            const int m = s > 0.f;
            out[g] = m ? s : 0.f;
            for (int k = 0; k < 4; ++k) out[(size_t)(1 + k) * H + g] = m ? tk[k] : 0.f;
        }
    }
    const float* aL = act + nl * NR * H;
    for (int o = 0; o < 4; ++o) {
        float s = b2[o];
        for (int h = 0; h < H; ++h) s += W2[o * H + h] * aL[h];
        y[o] = s;
        for (int k = 0; k < 4; ++k) {
            float j = 0.f;
            for (int h = 0; h < H; ++h) j = fmaf(W2[o * H + h], aL[(size_t)(1 + k) * H + h], j);
            J[o * 4 + k] = j;
        }
    }
}

static void point_d(int H, int L, const double* th, const double c[4], double* act, double y[4], double* J) {
    const size_t nl = (size_t)(L - 1), HH = (size_t)H * H;
    const double *W1 = th, *b1 = th + 4 * H, *Wh = th + 5 * H, *bh = Wh + nl * HH, *W2 = bh + nl * H, *b2 = W2 + 4 * H;
    for (int h = 0; h < H; ++h) {
        double s = b1[h];
        for (int k = 0; k < 4; ++k) s += W1[h * 4 + k] * c[k];
        const int m = s > 0.0;
        act[h] = m ? s : 0.0;
        for (int k = 0; k < 4; ++k) act[(size_t)(1 + k) * H + h] = m ? W1[h * 4 + k] : 0.0;
    }
    for (size_t l = 0; l < nl; ++l) {
        const double *W = Wh + l * HH, *in = act + l * NR * H;
        double* out = act + (l + 1) * NR * H;
        for (int g = 0; g < H; ++g) {
            double s = bh[l * H + g], tk[4] = {0.0, 0.0, 0.0, 0.0};
            for (int h = 0; h < H; ++h) {
                s += W[(size_t)g * H + h] * in[h];
                for (int k = 0; k < 4; ++k) tk[k] += W[(size_t)g * H + h] * in[(size_t)(1 + k) * H + h];
            }
            const int m = s > 0.0;
            out[g] = m ? s : 0.0;
            for (int k = 0; k < 4; ++k) out[(size_t)(1 + k) * H + g] = m ? tk[k] : 0.0;
        }
    }
    const double* aL = act + nl * NR * H;
    for (int o = 0; o < 4; ++o) {
        double s = b2[o];
        for (int k = 0; k < 4; ++k) J[o * 4 + k] = 0.0;
        for (int h = 0; h < H; ++h) {
            s += W2[o * H + h] * aL[h];
            for (int k = 0; k < 4; ++k) J[o * 4 + k] += W2[o * H + h] * aL[(size_t)(1 + k) * H + h];
        }
        y[o] = s;
    }
}

/* One point of the network in either mode (theta in double; the faithful mode rounds it and c to float). */
void oracle_deep_tangent_point(int H, int L, const double* theta, int all_double, const double c[4], double y[4], double J[16]) {
    const size_t NG = dt_len(H, L);
    if (all_double) {
        double* act = (double*)malloc(sizeof(double) * (size_t)L * NR * H);
        point_d(H, L, theta, c, act, y, J);
        free(act);
        return;
    }
    float* th = (float*)malloc(sizeof(float) * NG);
    float* act = (float*)malloc(sizeof(float) * (size_t)L * NR * H);
    for (size_t i = 0; i < NG; ++i) th[i] = (float)theta[i];
    const float cf[4] = {(float)c[0], (float)c[1], (float)c[2], (float)c[3]};
    float yf[4], Jf[16];
    point_f(H, L, th, cf, act, yf, Jf);
    for (int o = 0; o < 4; ++o) y[o] = yf[o];
    for (int i = 0; i < 16; ++i) J[i] = Jf[i];
    free(th);
    free(act);
}

/* The loss sums (and optionally the residuals, the faithful outputs y[N*4] and the gradient) over the whole grid.
 * theta: the parameters in double (the faithful mode rounds them to float, which is exact for fp32 weights). */
int oracle_deep_tangent_loss_grad(const oracle_grid* g, int H, int L, int m1p1, const double* theta, float t, float w_sigma,
                                  float w_u, int all_double, double* acc_s, double* acc_u, float* Rs, float* Rx, float* Ry,
                                  float* Rz, float* Y, double* grad) {
    const int nx = g->nx, ny = g->ny, nz = g->nz;
    const size_t N = (size_t)nx * ny * nz;
    if (!N || L < 1) return -1;
    const size_t NG = dt_len(H, L), nl = (size_t)(L - 1), HH = (size_t)H * H;
    float* th_f = (float*)malloc(sizeof(float) * NG);
    for (size_t i = 0; i < NG; ++i) th_f[i] = (float)theta[i];
    const double* th = theta;
    const double *Wh = th + 5 * H, *W2 = th + 5 * H + nl * (HH + H);
    float* af = (float*)malloc(sizeof(float) * (size_t)L * NR * H);
    double* ad = (double*)malloc(sizeof(double) * (size_t)L * NR * H);
    double* da = (double*)malloc(sizeof(double) * NR * H);   /* row adjoints of the current layer's output */
    double* dp = (double*)malloc(sizeof(double) * NR * H);
    if (grad)
        for (size_t i = 0; i < NG; ++i) grad[i] = 0.0;
    double *dW1 = grad, *db1 = grad ? grad + 4 * H : 0, *dWh = grad ? grad + 5 * H : 0, *dbh = grad ? dWh + nl * HH : 0;
    double *dW2 = grad ? dbh + nl * H : 0, *db2 = grad ? dW2 + 4 * H : 0;
    const double f = m1p1 ? 2.0 : 1.0;
    const double s[3] = {nx > 1 ? f / ((double)(nx - 1) * (double)g->hx) : 0.0, ny > 1 ? f / ((double)(ny - 1) * (double)g->hy) : 0.0,
                         nz > 1 ? f / ((double)(nz - 1) * (double)g->hz) : 0.0};
    const float ct = m1p1 ? t : t + 0.5f; /* src/mlp_grid.cpp:38 */
    double as = 0.0, au = 0.0;
    size_t i = 0;
    for (int z = 0; z < nz; ++z)
        for (int yy = 0; yy < ny; ++yy)
            for (int x = 0; x < nx; ++x, ++i) {
                const float cf[4] = {axis_coord(x, nx, m1p1), axis_coord(yy, ny, m1p1), axis_coord(z, nz, m1p1), ct};
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
                        if (Y) Y[i * 4 + o] = yf[o];
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
                if (Rs) { Rs[i] = (float)R[0]; Rx[i] = (float)R[1]; Ry[i] = (float)R[2]; Rz[i] = (float)R[3]; }
                as += R[0] * R[0];
                au += R[1] * R[1] + R[2] * R[2] + R[3] * R[3];
                if (!grad) continue;
                /* output seeds (DESIGN section 4.6.1) */
                double gb[4];
                for (int o = 0; o < 4; ++o) {
                    const float w = o == 0 ? w_sigma : w_u;
                    gb[o] = all_double ? 2.0 * (double)w / (double)N * R[o] : (double)((2.f * w / (float)N) * (float)R[o]);
                }
                double seed[NR][4]; /* row r: value row y_bar, tangent row k: J_bar[:,k] */
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
