/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the data-fit loss of deeper networks at arbitrary points
 * (tests/test_deep_data.py compiles it into a temporary shared library):
 *   acc = sum_i sum_o lam[o] (y_io - target_io)^2,  L_d = acc / n_norm,  grad = dL_d / d(every layer's weights)
 * for In = 4 -> H -> ... -> H -> Out = 4 with L >= 1 hidden layers.  PARITY UNPINNED (no reference counterpart).
 * Two modes:
 *   all_double = 0  forward by the strict-fp32 deep MLP (oracle_mlp_forward_deep's arithmetic, oracle/oracle.c: from the
 *                   bias, + W[g,h]*a[h] for h ascending, separately rounded multiply and add), seeds
 *                   y_bar_o = float(2 lam_o / n_norm) * (y_o - target_o) in fp32, the weighted sum in double, the adjoint
 *                   in double.  This is what the CUDA kernel is compared with.
 *   all_double = 1  everything in double: the function whose central finite differences pin the adjoint.
 * Parameters theta and gradient in the argument order of physad_set_weights_deep (doubles; the fp32 mode rounds theta):
 *   W1[H*4] | b1[H] | Wh[(L-1)*H*H, row-major [out][in]] | bh[(L-1)*H] | W2[4*H] | b2[4]
 * lam NULL: 1/4 each.  y (optional): the fp32 mode's outputs [B][4].
 */
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

static size_t plen(int H, int L) { return (size_t)9 * H + 4 + (size_t)(L - 1) * ((size_t)H * H + H); }

int oracle_data_loss_grad_deep(int H, int L, const double* theta, const float* x, const float* target, size_t B,
                               const float* lam_in, size_t n_norm, int all_double, double* acc_out, double* grad, float* y_out) {
    if (H < 1 || L < 1 || n_norm == 0) return -1;
    const size_t P = plen(H, L), nl = (size_t)(L - 1), HH = (size_t)H * H;
    const size_t oW1 = 0, ob1 = 4 * (size_t)H, oWh = 5 * (size_t)H, obh = oWh + nl * HH, oW2 = obh + nl * H, ob2 = oW2 + 4 * (size_t)H;
    float lam[4] = {0.25f, 0.25f, 0.25f, 0.25f};
    if (lam_in) memcpy(lam, lam_in, sizeof(lam));
    float* thf = (float*)malloc(sizeof(float) * P);
    double* a = (double*)malloc(sizeof(double) * (size_t)L * H);   /* activations of hidden layers 1..L (post-ReLU) */
    float* af = (float*)malloc(sizeof(float) * (size_t)L * H);
    double* da = (double*)malloc(sizeof(double) * H);
    double* dp = (double*)malloc(sizeof(double) * H);
    for (size_t e = 0; e < P; ++e) { thf[e] = (float)theta[e]; grad[e] = 0.0; }
    double acc = 0.0;
    for (size_t i = 0; i < B; ++i) {
        const float* xi = x + 4 * i;
        const float* ti = target + 4 * i;
        double dy[4];
        if (!all_double) {
            const float *W1 = thf + oW1, *b1 = thf + ob1, *Wh = thf + oWh, *bh = thf + obh, *W2 = thf + oW2, *b2 = thf + ob2;
            for (int h = 0; h < H; ++h) {
                float s = b1[h];
                for (int k = 0; k < 4; ++k) s += W1[h * 4 + k] * xi[k];
                af[h] = s > 0.f ? s : 0.f;
            }
            for (size_t l = 0; l < nl; ++l)
                for (int g = 0; g < H; ++g) {
                    float s = bh[l * H + g];
                    for (int h = 0; h < H; ++h) s += Wh[l * HH + (size_t)g * H + h] * af[l * H + h];
                    af[(l + 1) * H + g] = s > 0.f ? s : 0.f;
                }
            for (int o = 0; o < 4; ++o) {
                float s = b2[o];
                for (int h = 0; h < H; ++h) s += W2[o * H + h] * af[nl * H + h];
                if (y_out) y_out[4 * i + o] = s;
                const double e = (double)s - (double)ti[o];
                acc += (double)lam[o] * (e * e);
                const float coef = (float)(2.0 * (double)lam[o] / (double)n_norm);
                const float d = s - ti[o];
                const float yb = coef * d;
                dy[o] = (double)yb;
            }
            for (size_t q = 0; q < (size_t)L * H; ++q) a[q] = (double)af[q];
        } else {
            const double *W1 = theta + oW1, *b1 = theta + ob1, *Wh = theta + oWh, *bh = theta + obh, *W2 = theta + oW2, *b2 = theta + ob2;
            for (int h = 0; h < H; ++h) {
                double s = b1[h];
                for (int k = 0; k < 4; ++k) s += W1[h * 4 + k] * (double)xi[k];
                a[h] = s > 0.0 ? s : 0.0;
            }
            for (size_t l = 0; l < nl; ++l)
                for (int g = 0; g < H; ++g) {
                    double s = bh[l * H + g];
                    for (int h = 0; h < H; ++h) s += Wh[l * HH + (size_t)g * H + h] * a[l * H + h];
                    a[(l + 1) * H + g] = s > 0.0 ? s : 0.0;
                }
            for (int o = 0; o < 4; ++o) {
                double s = b2[o];
                for (int h = 0; h < H; ++h) s += W2[o * H + h] * a[nl * H + h];
                const double e = s - (double)ti[o];
                acc += (double)lam[o] * (e * e);
                dy[o] = 2.0 * (double)lam[o] / (double)n_norm * e;
            }
        }
        /* adjoint in double, weights as the forward used them */
        const double* W2d = theta + oW2;
        for (int o = 0; o < 4; ++o) {
            grad[ob2 + o] += dy[o];
            for (int h = 0; h < H; ++h) grad[oW2 + (size_t)o * H + h] += dy[o] * a[nl * H + h];
        }
        for (int h = 0; h < H; ++h) {
            double s = 0.0;
            for (int o = 0; o < 4; ++o) s += (all_double ? W2d[o * H + h] : (double)thf[oW2 + (size_t)o * H + h]) * dy[o];
            da[h] = s;
        }
        for (size_t l = nl; l-- > 0;) {   /* hidden -> hidden layer l: a_{l+1} = relu(W a_l + b) */
            for (int g = 0; g < H; ++g) da[g] = a[(l + 1) * H + g] > 0.0 ? da[g] : 0.0;
            for (int g = 0; g < H; ++g) {
                grad[obh + l * H + g] += da[g];
                for (int h = 0; h < H; ++h) grad[oWh + l * HH + (size_t)g * H + h] += da[g] * a[l * H + h];
            }
            for (int h = 0; h < H; ++h) {
                double s = 0.0;
                for (int g = 0; g < H; ++g) {
                    const size_t e = oWh + l * HH + (size_t)g * H + h;
                    s += (all_double ? theta[e] : (double)thf[e]) * da[g];
                }
                dp[h] = s;
            }
            memcpy(da, dp, sizeof(double) * H);
        }
        for (int h = 0; h < H; ++h) {
            const double dz = a[h] > 0.0 ? da[h] : 0.0;
            grad[ob1 + h] += dz;
            for (int k = 0; k < 4; ++k) grad[oW1 + (size_t)h * 4 + k] += dz * (double)xi[k];
        }
    }
    *acc_out = acc;
    free(thf); free(a); free(af); free(da); free(dp);
    return 0;
}
