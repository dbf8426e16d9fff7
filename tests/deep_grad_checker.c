/*
 * TEST INFRASTRUCTURE ONLY -- CPU checker for the closed loop of deeper networks (tests/test_deep_grad.py compiles it
 * into a temporary shared library): d(L_sigma + L_u) / d(every layer's weights) of the finite-difference loss for
 * In = 4 -> H -> ... -> H -> Out = 4 with L >= 1 hidden layers.
 *
 * PARITY UNPINNED, like oracle/oracle_grad.c, whose helpers it reuses by inclusion (grid, coordinates, the neighbour
 * rule, the transposed central difference, the slice times) and whose two modes it keeps:
 *   all_double = 0  fields by the strict-fp32 deep MLP (oracle_mlp_forward_deep's arithmetic, oracle/oracle.c),
 *                   residuals rounded to float, g = (2w/float(N))*R in fp32; the adjoint runs in double.  This is what
 *                   the CUDA kernel is compared with.
 *   all_double = 1  everything in double: the function whose central finite differences pin the adjoint.
 * Parameters and gradient in the argument order of physad_set_weights_deep:
 *   W1[H*4] | b1[H] | Wh[(L-1)*H*H, row-major [out][in]] | bh[(L-1)*H] | W2[4*H] | b2[4]
 * For L = 1 the gradient equals oracle_phys_loss_grad's bit for bit (the test checks it).
 */
#include "../oracle/oracle_grad.c"

/* Deep network, L >= 1 hidden layers, parameters in the gradient layout
 *   W1[H*4] | b1[H] | Wh[(L-1)*H*H, row-major [out][in]] | bh[(L-1)*H] | W2[4*H] | b2[4].
 * act[l*H + h]: post-ReLU activation of hidden layer l+1 (a > 0 iff the pre-activation is).  Every layer is the
 * reference's layer rule (from the bias, + W[g,h]*a[h] for h ascending); the fp32 form is oracle_mlp_forward_deep's
 * arithmetic (oracle.c), the double form the same formulas in double. */
static void mlp_point_deep_f(int H, int L, const float* th, const float x[4], float* act, double y[4]) {
    const size_t nl = (size_t)(L - 1), HH = (size_t)H * H;
    const float *W1 = th, *b1 = th + 4 * H, *Wh = th + 5 * H, *bh = Wh + nl * HH, *W2 = bh + nl * H, *b2 = W2 + 4 * H;
    for (int h = 0; h < H; ++h) {
        float s = b1[h];
        for (int k = 0; k < 4; ++k) s += W1[h * 4 + k] * x[k];
        act[h] = s > 0.f ? s : 0.f;
    }
    for (size_t l = 0; l < nl; ++l)
        for (int g2 = 0; g2 < H; ++g2) {
            float s = bh[l * H + g2];
            for (int h = 0; h < H; ++h) s += Wh[l * HH + (size_t)g2 * H + h] * act[l * H + h];
            act[(l + 1) * H + g2] = s > 0.f ? s : 0.f;
        }
    for (int o = 0; o < 4; ++o) {
        float s = b2[o];
        for (int h = 0; h < H; ++h) s += W2[o * H + h] * act[nl * H + h];
        y[o] = (double)s;
    }
}

static void mlp_point_deep_d(int H, int L, const double* th, const float x[4], double* act, double y[4]) {
    const size_t nl = (size_t)(L - 1), HH = (size_t)H * H;
    const double *W1 = th, *b1 = th + 4 * H, *Wh = th + 5 * H, *bh = Wh + nl * HH, *W2 = bh + nl * H, *b2 = W2 + 4 * H;
    for (int h = 0; h < H; ++h) {
        double s = b1[h];
        for (int k = 0; k < 4; ++k) s += W1[h * 4 + k] * (double)x[k];
        act[h] = s > 0.0 ? s : 0.0;
    }
    for (size_t l = 0; l < nl; ++l)
        for (int g2 = 0; g2 < H; ++g2) {
            double s = bh[l * H + g2];
            for (int h = 0; h < H; ++h) s += Wh[l * HH + (size_t)g2 * H + h] * act[l * H + h];
            act[(l + 1) * H + g2] = s > 0.0 ? s : 0.0;
        }
    for (int o = 0; o < 4; ++o) {
        double s = b2[o];
        for (int h = 0; h < H; ++h) s += W2[o * H + h] * act[nl * H + h];
        y[o] = s;
    }
}

static size_t deep_len(int H, int L) { return (size_t)9 * H + 4 + (size_t)(L - 1) * ((size_t)H * H + H); }

/* forward_all of oracle_grad.c with the deep point functions: F[(s*4 + c)*N + i], R[c*N + i], sums of squares. */
static void forward_all_deep(const model* m, int L, double* F, double* R, double* acc_s, double* acc_u) {
    const oracle_grid* g = m->g;
    const int nx = g->nx, ny = g->ny, nz = g->nz, per = g->periodic, H = m->H;
    const size_t N = (size_t)nx * ny * nz;
    float* zf = (float*)malloc(sizeof(float) * (size_t)L * H);
    double* zd = (double*)malloc(sizeof(double) * (size_t)L * H);
    for (int s = 0; s < 3; ++s)
        for (size_t i = 0; i < N; ++i) {
            float x[4];
            double y[4];
            point_coords(m, i, s, x);
            if (m->all_double) mlp_point_deep_d(H, L, m->th_d, x, zd, y);
            else mlp_point_deep_f(H, L, m->th_f, x, zf, y);
            for (int c = 0; c < 4; ++c) F[((size_t)s * 4 + c) * N + i] = y[c];
        }
    free(zf);
    free(zd);
    const double i2t = 1.0 / (2.0 * (double)g->dt), i2x = 1.0 / (2.0 * (double)g->hx);
    const double i2y = 1.0 / (2.0 * (double)g->hy), i2z = 1.0 / (2.0 * (double)g->hz);
    const double *Fm = F, *F0 = F + 4 * N, *Fp = F + 8 * N;
    double as = 0.0, au = 0.0;
#define LIN(X, Y, Z) ((size_t)(((Z) * ny + (Y)) * nx + (X)))
    for (int z = 0; z < nz; ++z)
        for (int y = 0; y < ny; ++y)
            for (int x = 0; x < nx; ++x) {
                const size_t i = LIN(x, y, z);
                const size_t xp = LIN(nb(x + 1, nx, per), y, z), xm = LIN(nb(x - 1, nx, per), y, z);
                const size_t yp = LIN(x, nb(y + 1, ny, per), z), ym = LIN(x, nb(y - 1, ny, per), z);
                const size_t zp = LIN(x, y, nb(z + 1, nz, per)), zm = LIN(x, y, nb(z - 1, nz, per));
                double dt_[4], gr[4][3];
                for (int c = 0; c < 4; ++c) {
                    const double* f = F0 + (size_t)c * N;
                    dt_[c] = (Fp[(size_t)c * N + i] - Fm[(size_t)c * N + i]) * i2t;
                    gr[c][0] = (f[xp] - f[xm]) * i2x;
                    gr[c][1] = (f[yp] - f[ym]) * i2y;
                    gr[c][2] = (f[zp] - f[zm]) * i2z;
                }
                const double u[3] = {F0[N + i], F0[2 * N + i], F0[3 * N + i]};
                const double div = gr[1][0] + gr[2][1] + gr[3][2];
                const double adv_s = u[0] * gr[0][0] + u[1] * gr[0][1] + u[2] * gr[0][2];
                double r[4];
                r[0] = dt_[0] + adv_s + F0[i] * div; /* src/phys_cpu.cpp:103 */
                for (int c = 1; c < 4; ++c) r[c] = dt_[c] + (u[0] * gr[c][0] + u[1] * gr[c][1] + u[2] * gr[c][2]); /* :104-106 */
                for (int c = 0; c < 4; ++c) {
                    if (!m->all_double) r[c] = (double)(float)r[c];
                    R[(size_t)c * N + i] = r[c];
                }
                as += r[0] * r[0];
                au += r[1] * r[1] + r[2] * r[2] + r[3] * r[3];
            }
#undef LIN
    *acc_s = as;
    *acc_u = au;
}

/* ---- the loss and its gradient -----------------------------------------------------------------------------------------
 * Same two modes as oracle_phys_loss_grad.  The stencil adjoint is that function's, restated; the MLP backward runs
 * through every layer: delta_a_L = W2^T A, then per hidden layer delta_z = delta_a (.) (a > 0), dW += delta_z a_prev^T,
 * db += delta_z, delta_a_prev = W^T delta_z; layer 1 against the point's coordinates (x, y, z, t_slice). */
int oracle_phys_loss_double_deep(const oracle_grid* g, int H, int L, int m1p1, const double* theta, float t, float dt,
                                 float w_sigma, float w_u, double* loss_sigma, double* loss_u) {
    const size_t N = (size_t)g->nx * g->ny * g->nz;
    if (!N || L < 1) return -1;
    model m = {g, H, m1p1, 1, 0, theta, {0, 0, 0}};
    const float off = m1p1 ? 0.f : 0.5f;
    m.ts[0] = (t - dt) + off; m.ts[1] = t + off; m.ts[2] = (t + dt) + off;
    double* F = (double*)malloc(sizeof(double) * 12 * N);
    double* R = (double*)malloc(sizeof(double) * 4 * N);
    double as, au;
    forward_all_deep(&m, L, F, R, &as, &au);
    *loss_sigma = (double)w_sigma * as / (double)N;
    *loss_u = (double)w_u * au / (double)N;
    free(F);
    free(R);
    return 0;
}

int oracle_phys_loss_grad_deep(const oracle_grid* g, int H, int L, int m1p1, const float* W1, const float* b1, const float* Wh,
                               const float* bh, const float* W2, const float* b2, float t, float dt, float w_sigma, float w_u,
                               int all_double, double* loss_sigma, double* loss_u, double* grad) {
    const int nx = g->nx, ny = g->ny, nz = g->nz, per = g->periodic;
    const size_t N = (size_t)nx * ny * nz;
    if (!N || L < 1) return -1;
    const size_t NG = deep_len(H, L), nl = (size_t)(L - 1), HH = (size_t)H * H;
    float* th_f = (float*)malloc(sizeof(float) * NG);
    double* th_d = (double*)malloc(sizeof(double) * NG);
    memcpy(th_f, W1, sizeof(float) * 4 * H);
    memcpy(th_f + 4 * H, b1, sizeof(float) * H);
    if (nl) {
        memcpy(th_f + 5 * H, Wh, sizeof(float) * nl * HH);
        memcpy(th_f + 5 * H + nl * HH, bh, sizeof(float) * nl * H);
    }
    memcpy(th_f + 5 * H + nl * (HH + H), W2, sizeof(float) * 4 * H);
    memcpy(th_f + 9 * H + nl * (HH + H), b2, sizeof(float) * 4);
    for (size_t i = 0; i < NG; ++i) th_d[i] = (double)th_f[i];
    model m = {g, H, m1p1, all_double, th_f, th_d, {0, 0, 0}};
    const float off = m1p1 ? 0.f : 0.5f;
    m.ts[0] = (t - dt) + off; m.ts[1] = t + off; m.ts[2] = (t + dt) + off;

    double* F = (double*)malloc(sizeof(double) * 12 * N);
    double* R = (double*)malloc(sizeof(double) * 4 * N);
    double as, au;
    forward_all_deep(&m, L, F, R, &as, &au);
    if (loss_sigma) *loss_sigma = (double)w_sigma * as / (double)N;
    if (loss_u) *loss_u = (double)w_u * au / (double)N;

    double* G = (double*)malloc(sizeof(double) * 4 * N);
    for (int c = 0; c < 4; ++c) {
        const float w = c == 0 ? w_sigma : w_u;
        if (all_double) {
            const double k = 2.0 * (double)w / (double)N;
            for (size_t i = 0; i < N; ++i) G[(size_t)c * N + i] = k * R[(size_t)c * N + i];
        } else {
            const float k = 2.f * w / (float)N;
            for (size_t i = 0; i < N; ++i) G[(size_t)c * N + i] = (double)(k * (float)R[(size_t)c * N + i]);
        }
    }
    const double* F0 = F + 4 * N;
    double* Cf = (double*)malloc(sizeof(double) * 12 * N);
    for (int j = 0; j < 3; ++j)
        for (size_t p = 0; p < N; ++p) {
            const double uj = F0[(size_t)(j + 1) * N + p];
            Cf[((size_t)j * 4 + 0) * N + p] = G[p] * uj;
            for (int i = 0; i < 3; ++i)
                Cf[((size_t)j * 4 + i + 1) * N + p] = G[(size_t)(i + 1) * N + p] * uj + (i == j ? G[p] * F0[p] : 0.0);
        }
    const double i2t = 1.0 / (2.0 * (double)g->dt);
    const double i2h[3] = {1.0 / (2.0 * (double)g->hx), 1.0 / (2.0 * (double)g->hy), 1.0 / (2.0 * (double)g->hz)};
    for (size_t i = 0; i < NG; ++i) grad[i] = 0.0;
    double *dW1 = grad, *db1 = grad + 4 * H, *dWh = grad + 5 * H, *dbh = dWh + nl * HH, *dW2 = dbh + nl * H, *db2 = dW2 + 4 * H;
    const double *tW2 = th_d + 5 * H + nl * (HH + H), *tWh = th_d + 5 * H;
    float* af = (float*)malloc(sizeof(float) * (size_t)L * H);
    double* ad = (double*)malloc(sizeof(double) * (size_t)L * H);
    double* da = (double*)malloc(sizeof(double) * H);
    double* dz = (double*)malloc(sizeof(double) * H);
#define LIN(X, Y, Z) ((size_t)(((Z) * ny + (Y)) * nx + (X)))
    for (int z = 0; z < nz; ++z)
        for (int y = 0; y < ny; ++y)
            for (int x = 0; x < nx; ++x) {
                const size_t q = LIN(x, y, z);
                const size_t xp = LIN(nb(x + 1, nx, per), y, z), xm = LIN(nb(x - 1, nx, per), y, z);
                const size_t yp = LIN(x, nb(y + 1, ny, per), z), ym = LIN(x, nb(y - 1, ny, per), z);
                const size_t zp = LIN(x, y, nb(z + 1, nz, per)), zm = LIN(x, y, nb(z - 1, nz, per));
                const size_t ip[3] = {xp, yp, zp}, im[3] = {xm, ym, zm};
                double gr[4][3];
                for (int c = 0; c < 4; ++c)
                    for (int j = 0; j < 3; ++j) gr[c][j] = (F0[(size_t)c * N + ip[j]] - F0[(size_t)c * N + im[j]]) * i2h[j];
                double A[3][4];
                A[1][0] = G[q] * (gr[1][0] + gr[2][1] + gr[3][2]);
                for (int j = 0; j < 3; ++j)
                    A[1][j + 1] = G[q] * gr[0][j] + G[N + q] * gr[1][j] + G[2 * N + q] * gr[2][j] + G[3 * N + q] * gr[3][j];
                const int qi[3] = {x, y, z}, nn[3] = {nx, ny, nz};
                const size_t stride[3] = {1, (size_t)nx, (size_t)nx * ny};
                for (int j = 0; j < 3; ++j) {
                    const size_t base = q - (size_t)qi[j] * stride[j];
                    for (int c = 0; c < 4; ++c)
                        A[1][c] += i2h[j] * transposed_diff(Cf + ((size_t)j * 4 + c) * N, base, stride[j], qi[j], nn[j], per);
                }
                for (int c = 0; c < 4; ++c) {
                    A[2][c] = G[(size_t)c * N + q] * i2t;
                    A[0][c] = -A[2][c];
                }
                for (int s = 0; s < 3; ++s) {
                    float xin[4];
                    double yy[4];
                    point_coords(&m, q, s, xin);
                    if (all_double) mlp_point_deep_d(H, L, th_d, xin, ad, yy);
                    else {
                        mlp_point_deep_f(H, L, th_f, xin, af, yy);
                        for (size_t i = 0; i < (size_t)L * H; ++i) ad[i] = (double)af[i];
                    }
                    for (int o = 0; o < 4; ++o) db2[o] += A[s][o];
                    const double* aL = ad + nl * H;
                    for (int h = 0; h < H; ++h) {
                        double v = 0.0;
                        for (int o = 0; o < 4; ++o) {
                            dW2[o * H + h] += A[s][o] * aL[h];
                            v += tW2[o * H + h] * A[s][o];
                        }
                        da[h] = v;
                    }
                    for (size_t l = nl; l >= 1; --l) {   /* hidden layer l+1 (weights Wh[l-1]) */
                        const double *a_out = ad + l * H, *a_in = ad + (l - 1) * H, *W = tWh + (l - 1) * HH;
                        for (int g2 = 0; g2 < H; ++g2) {
                            dz[g2] = a_out[g2] > 0.0 ? da[g2] : 0.0;
                            dbh[(l - 1) * H + g2] += dz[g2];
                            for (int h = 0; h < H; ++h) dWh[(l - 1) * HH + (size_t)g2 * H + h] += dz[g2] * a_in[h];
                        }
                        for (int h = 0; h < H; ++h) {
                            double v = 0.0;
                            for (int g2 = 0; g2 < H; ++g2) v += W[(size_t)g2 * H + h] * dz[g2];
                            da[h] = v;
                        }
                    }
                    for (int h = 0; h < H; ++h) {
                        const double d = ad[h] > 0.0 ? da[h] : 0.0;
                        db1[h] += d;
                        for (int k = 0; k < 4; ++k) dW1[h * 4 + k] += d * (double)xin[k];
                    }
                }
            }
#undef LIN
    free(af); free(ad); free(da); free(dz); free(Cf); free(G); free(R); free(F); free(th_f); free(th_d);
    return 0;
}
