/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the periodic-pair loss of deeper networks
 * (tests/test_deep_pair.py compiles it into a temporary shared library, -ffp-contract=off):
 *   acc = sum_i sum_o lam[o] (y(p_i)_o - y(q_i)_o)^2,  L_p = acc / n_norm,  grad = dL_p / d(every layer's weights)
 * for In = 4 -> H -> ... -> H -> Out = 4 with L >= 1 hidden layers, x = B pairs [B][2][4] (p_i, q_i).
 * PARITY UNPINNED (no reference counterpart).  Its own forward and adjoint per point; deep_data_checker.c (included below)
 * is in the same library so that the tests can tie the two checkers together.  Two modes:
 *   all_double = 0  forward by the strict-fp32 deep MLP (oracle_mlp_forward_deep's arithmetic), seeds as the CUDA kernel
 *                   forms them: y_bar(p)_o = float(2 lam_o / n_norm) * (y(p)_o - y(q)_o) in fp32 and y_bar(q) = -y_bar(p),
 *                   the weighted sum in double, the adjoint in double.  This is what the CUDA kernel is compared with.
 *   all_double = 1  everything in double: the function whose central finite differences pin the adjoint.
 * Parameters theta and gradient in the argument order of physad_set_weights_deep (deep_data_checker.c's layout).
 * lam NULL: 1/4 each.  y (optional): the fp32 mode's outputs [B][2][4].
 */
#include "deep_data_checker.c"

typedef struct {
    int H, L, all_double;
    const double* theta;
    const float* thf;
} pair_net;

/* a[L*H] (post-ReLU activations, as doubles) and the outputs of one point */
static void pair_forward(const pair_net* n, const float* xi, double* a, float* af, double y[4], float yf[4]) {
    const int H = n->H;
    const size_t nl = (size_t)(n->L - 1), HH = (size_t)H * H;
    const size_t oWh = 5 * (size_t)H, obh = oWh + nl * HH, oW2 = obh + nl * H, ob2 = oW2 + 4 * (size_t)H;
    if (!n->all_double) {
        const float *W1 = n->thf, *b1 = n->thf + 4 * H, *Wh = n->thf + oWh, *bh = n->thf + obh, *W2 = n->thf + oW2, *b2 = n->thf + ob2;
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
            yf[o] = s;
            y[o] = (double)s;
        }
        for (size_t q = 0; q < (size_t)n->L * H; ++q) a[q] = (double)af[q];
    } else {
        const double* th = n->theta;
        const double *W1 = th, *b1 = th + 4 * H, *Wh = th + oWh, *bh = th + obh, *W2 = th + oW2, *b2 = th + ob2;
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
            y[o] = s;
            yf[o] = (float)s;
        }
    }
}

/* grad += d(dy . y(xi)) / d theta, in double, with the weights the forward used */
static void pair_backward(const pair_net* n, const float* xi, const double* a, const double dy[4], double* grad, double* da,
                          double* dp) {
    const int H = n->H;
    const size_t nl = (size_t)(n->L - 1), HH = (size_t)H * H;
    const size_t ob1 = 4 * (size_t)H, oWh = 5 * (size_t)H, obh = oWh + nl * HH, oW2 = obh + nl * H, ob2 = oW2 + 4 * (size_t)H;
#define PAIR_W(e) (n->all_double ? n->theta[e] : (double)n->thf[e])
    for (int o = 0; o < 4; ++o) {
        grad[ob2 + o] += dy[o];
        for (int h = 0; h < H; ++h) grad[oW2 + (size_t)o * H + h] += dy[o] * a[nl * H + h];
    }
    for (int h = 0; h < H; ++h) {
        double s = 0.0;
        for (int o = 0; o < 4; ++o) s += PAIR_W(oW2 + (size_t)o * H + h) * dy[o];
        da[h] = s;
    }
    for (size_t l = nl; l-- > 0;) {
        for (int g = 0; g < H; ++g) da[g] = a[(l + 1) * H + g] > 0.0 ? da[g] : 0.0;
        for (int g = 0; g < H; ++g) {
            grad[obh + l * H + g] += da[g];
            for (int h = 0; h < H; ++h) grad[oWh + l * HH + (size_t)g * H + h] += da[g] * a[l * H + h];
        }
        for (int h = 0; h < H; ++h) {
            double s = 0.0;
            for (int g = 0; g < H; ++g) s += PAIR_W(oWh + l * HH + (size_t)g * H + h) * da[g];
            dp[h] = s;
        }
        memcpy(da, dp, sizeof(double) * H);
    }
    for (int h = 0; h < H; ++h) {
        const double dz = a[h] > 0.0 ? da[h] : 0.0;
        grad[ob1 + h] += dz;
        for (int k = 0; k < 4; ++k) grad[(size_t)h * 4 + k] += dz * (double)xi[k];
    }
#undef PAIR_W
}

int oracle_pair_loss_grad_deep(int H, int L, const double* theta, const float* x, size_t B, const float* lam_in,
                               size_t n_norm, int all_double, double* acc_out, double* grad, float* y_out) {
    if (H < 1 || L < 1 || n_norm == 0) return -1;
    const size_t P = plen(H, L), LH = (size_t)L * H;
    float lam[4] = {0.25f, 0.25f, 0.25f, 0.25f};
    if (lam_in) memcpy(lam, lam_in, sizeof(lam));
    float* thf = (float*)malloc(sizeof(float) * P);
    double* a = (double*)malloc(sizeof(double) * 2 * LH);
    float* af = (float*)malloc(sizeof(float) * LH);
    double* da = (double*)malloc(sizeof(double) * H);
    double* dp = (double*)malloc(sizeof(double) * H);
    for (size_t e = 0; e < P; ++e) { thf[e] = (float)theta[e]; grad[e] = 0.0; }
    const pair_net net = {H, L, all_double, theta, thf};
    double acc = 0.0;
    for (size_t i = 0; i < B; ++i) {
        const float *xp = x + 8 * i, *xq = xp + 4;
        double yp[4], yq[4], dy[4], dq[4];
        float fp[4], fq[4];
        pair_forward(&net, xp, a, af, yp, fp);
        pair_forward(&net, xq, a + LH, af, yq, fq);
        for (int o = 0; o < 4; ++o) {
            if (y_out) { y_out[8 * i + o] = fp[o]; y_out[8 * i + 4 + o] = fq[o]; }
            const double e = yp[o] - yq[o];
            acc += (double)lam[o] * (e * e);
            if (!all_double) {
                const float coef = (float)(2.0 * (double)lam[o] / (double)n_norm);
                const float d = fp[o] - fq[o];
                const float yb = coef * d;
                dy[o] = (double)yb;
            } else {
                dy[o] = 2.0 * (double)lam[o] / (double)n_norm * e;
            }
            dq[o] = -dy[o];
        }
        pair_backward(&net, xp, a, dy, grad, da, dp);
        pair_backward(&net, xq, a + LH, dq, grad, da, dp);
    }
    *acc_out = acc;
    free(thf); free(a); free(af); free(da); free(dp);
    return 0;
}
