// The deep data-fit kernels; see deep_data_kernels.cuh for what they compute.
//
// k_deep_data_grad<H> is k_deep_grad<H> (deep_grad_kernels.cu) with one row per point instead of three (point x time
// slice): the same tile geometry (256 threads, a warp owns 16 units of one row-block, a lane 6 rows; H = 128: 1 row-block
// of 192 rows, 64: 2, 32: 4), the same shared-memory layout and checkpoint area, the same backward.  What differs:
//   * a row's coordinates are the caller's point (one float4 load) and W1[h,3] * t is rounded per row, as in
//     k_mlp_deep's points mode, so the recomputed network is bit-identical to physad_mlp_forward_deep_dev's;
//   * the output layer is computed (k_deep_grad only needs the adjoint the physics kernels leave behind), with
//     k_mlp_deep's arithmetic and weights from the same kernel-parameter block;
//   * y_bar is formed here from the outputs and the targets, and L = 1 (no hidden -> hidden layer) is allowed.
// The hidden-layer weights are staged one layer at a time in one shared buffer exactly as in k_deep_grad.
// No FFMA2 anywhere: the forward keeps k_mlp_deep's un-contracted FMUL2 / FADD2, the backward uses scalar FFMA.
#include "deep_data_kernels.cuh"
#include "mlp_eval.cuh"

namespace physad {

namespace {

__device__ __forceinline__ unsigned smem_addr(const void* p) { return unsigned(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

constexpr int NT = DEEP_DATA_THREADS;
constexpr int GT = 16;          // units per warp
constexpr int PT = 6;           // rows (= points) per lane
constexpr int ROWS = 32 * PT;   // rows per row-block
constexpr int CH = 64;          // rows per staging chunk of the dW step

constexpr int cmax(int x, int y) { return x > y ? x : y; }

template <int H>
struct Geo {
    static constexpr int G = H / GT;               // warps per row-block
    static constexpr int RB = 8 / G;               // row-blocks per tile
    static constexpr int NROW = RB * ROWS;         // rows = points per tile
    static constexpr int ACT = RB * H * ROWS;      // floats of one layer's activations (24576 for every H)
    static constexpr int SCR = cmax(cmax(H * H, CH * (H + 1)), 4 * NROW);   // staging: dW chunk | y_bar / coords
    static constexpr size_t SMEM = (size_t(ACT) + 5 * H + H * H + SCR) * sizeof(float);
};

__host__ __device__ constexpr size_t grad_len(int H, int L) {
    return size_t(9) * H + 4 + size_t(L - 1) * (size_t(H) * H + H);
}

template <int H>
__global__ void __launch_bounds__(NT, 1) k_deep_data_grad(const __grid_constant__ MlpConst<H> w, const __grid_constant__ DeepDataArgs a) {
    using Q = Geo<H>;
    constexpr int G = Q::G, RB = Q::RB, NROW = Q::NROW, PTS_TILE = NROW, ACT = Q::ACT;
    extern __shared__ __align__(16) float smem[];
    float* s_act = smem;                                              // [RB][H][ROWS]
    float2* s_l1 = reinterpret_cast<float2*>(smem + ACT);             // [5][H/2] layer-1 pairs (as k_mlp_deep)
    float* s_w = smem + ACT + 5 * H;                                  // [H][H] one hidden layer, k_mlp_deep's layout
    float* s_scr = s_w + H * H;                                       // staging: [CH][H+1] | y_bar / coords [NROW] float4
    float4* s_row = reinterpret_cast<float4*>(s_scr);
    __shared__ double s_red[NT / 32][5];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rb = warp / G, g0 = (warp % G) * GT;
    const int L = a.hidden_layers, nl = L - 1;
    const long long n = a.n;
    const long long tiles = (n + PTS_TILE - 1) / PTS_TILE;

    const size_t P = grad_len(H, L);
    const size_t oW1 = 0, ob1 = 4 * H, oWh = 5 * H, obh = oWh + size_t(nl) * H * H, oW2 = obh + size_t(nl) * H, ob2 = oW2 + 4 * H;
    double* part = a.partials + size_t(blockIdx.x) * (P + 1);
    float* ck = a.ckpt + size_t(blockIdx.x) * L * ACT;
    for (size_t e = threadIdx.x; e < P + 1; e += NT) part[e] = 0.0;

    int wcur = -1;   // hidden layer whose weights are (being) staged in s_w
    auto load_layer = [&](int layer) {
        const float* src = a.wh + size_t(layer) * H * H;
        for (int i = threadIdx.x; i < H * H / 4; i += NT) cp_async16(s_w + 4 * i, src + 4 * i);
        cp_async_commit();
        wcur = layer;
    };
    for (int q = threadIdx.x; q < H / 2; q += NT) {
        const float4 ra = __ldg(reinterpret_cast<const float4*>(a.W1) + 2 * q), rb4 = __ldg(reinterpret_cast<const float4*>(a.W1) + 2 * q + 1);
        s_l1[q] = make_float2(__ldg(a.b1 + 2 * q), __ldg(a.b1 + 2 * q + 1));
        s_l1[H / 2 + q] = make_float2(rb4.x, ra.x);
        s_l1[2 * (H / 2) + q] = make_float2(rb4.y, ra.y);
        s_l1[3 * (H / 2) + q] = make_float2(rb4.z, ra.z);
        s_l1[4 * (H / 2) + q] = make_float2(ra.w, rb4.w);
    }
    double red[5] = {0.0, 0.0, 0.0, 0.0, 0.0};   // db2[4], sum lam (y - target)^2
    __syncthreads();

    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        if (nl > 0 && wcur != 0) load_layer(0);   // s_w is free: the previous tile's last contraction is behind a barrier
        // ================= forward ================================================================================
        // ---- layer 1 (k_mlp_deep's points-mode arithmetic) -> s_act and checkpoint 0 -----------------------------
        {
            float cx[PT], cy[PT], cz[PT], ct[PT];
#pragma unroll
            for (int j = 0; j < PT; ++j) {
                long long p = tile * PTS_TILE + rb * ROWS + lane * PT + j;
                if (p > n - 1) p = n - 1;   // tail tile: a valid point, its y_bar is zero
                const float4 c4 = __ldg(a.x + p);
                cx[j] = c4.x; cy[j] = c4.y; cz[j] = c4.z; ct[j] = c4.w;
            }
            const int off = (rb * H) * ROWS + lane * PT;
            float* dst = s_act + off;
            float* dck = ck + off;
#pragma unroll 2
            for (int q = 0; q < GT / 2; ++q) {
                const int qq = g0 / 2 + q;
                const float2 b1p = s_l1[qq], w0s = s_l1[H / 2 + qq], w1s = s_l1[2 * (H / 2) + qq], w2s = s_l1[3 * (H / 2) + qq];
                const float2 w3 = s_l1[4 * (H / 2) + qq];
#pragma unroll
                for (int j = 0; j < PT; ++j) {
                    const f32x2 sx = add2_rn_swapped(pack2(b1p), mul2_rn(pack2(w0s), bcast2(cx[j])));
                    const f32x2 sxy = add2_rn_swapped(sx, mul2_rn(pack2(w1s), bcast2(cy[j])));
                    const f32x2 sxyz = add2_rn_swapped(sxy, mul2_rn(pack2(w2s), bcast2(cz[j])));
                    const float2 pt = make_float2(__fmul_rn(w3.x, ct[j]), __fmul_rn(w3.y, ct[j]));
                    float v0, v1;
                    unpack2(add2_rn(sxyz, pack2(pt)), v0, v1);
                    v0 = relu_ref(v0); v1 = relu_ref(v1);
                    dst[(2 * qq) * ROWS + j] = v0;
                    dst[(2 * qq + 1) * ROWS + j] = v1;
                    dck[(2 * qq) * ROWS + j] = v0;
                    dck[(2 * qq + 1) * ROWS + j] = v1;
                }
            }
        }
        // ---- hidden -> hidden layers -> s_act and checkpoints 1..L-1 -------------------------------------------
        for (int l = 0; l < nl; ++l) {
            cp_async_wait_all();
            __syncthreads();   // layer l's weights have landed, its inputs are written
            const float* wbuf = s_w + g0;
            const float* arow = s_act + (rb * H) * ROWS + lane * PT;
            f32x2 q[PT][GT / 2];
            {
                const float* bl = a.bh + size_t(l) * H + g0;
#pragma unroll
                for (int p = 0; p < GT / 2; ++p) {
                    const float2 b = __ldg(reinterpret_cast<const float2*>(bl) + p);
#pragma unroll
                    for (int j = 0; j < PT; ++j) q[j][p] = pack2(b.x, b.y);
                }
            }
#pragma unroll 4
            for (int h = 0; h < H; ++h) {
                float av[PT];
                float4 wv[GT / 4];
#pragma unroll
                for (int j = 0; j < PT; j += 2) {
                    const float2 t = *reinterpret_cast<const float2*>(arow + h * ROWS + j);
                    av[j] = t.x; av[j + 1] = t.y;
                }
#pragma unroll
                for (int v = 0; v < GT / 4; ++v) wv[v] = *reinterpret_cast<const float4*>(wbuf + h * H + 4 * v);
#pragma unroll
                for (int j = 0; j < PT; ++j) {
                    const f32x2 aa = bcast2(av[j]);
#pragma unroll
                    for (int v = 0; v < GT / 4; ++v) {   // {W[g+1,h], W[g,h], W[g+3,h], W[g+2,h]}
                        q[j][2 * v] = add2_rn_swapped(q[j][2 * v], mul2_rn(aa, pack2(wv[v].x, wv[v].y)));
                        q[j][2 * v + 1] = add2_rn_swapped(q[j][2 * v + 1], mul2_rn(aa, pack2(wv[v].z, wv[v].w)));
                    }
                }
            }
            __syncthreads();   // every warp has read this layer's inputs and weights
            if (l + 1 < nl) load_layer(l + 1);   // the last forward layer's weights are the first backward layer's
            {
                const int off = (rb * H + g0) * ROWS + lane * PT;
                float* orow = s_act + off;
                float* ocK = ck + size_t(l + 1) * ACT + off;
#pragma unroll
                for (int p = 0; p < GT / 2; ++p) {
                    float lo[PT], hi[PT];
#pragma unroll
                    for (int j = 0; j < PT; ++j) {
                        unpack2(q[j][p], lo[j], hi[j]);
                        lo[j] = relu_ref(lo[j]); hi[j] = relu_ref(hi[j]);
                    }
#pragma unroll
                    for (int j = 0; j < PT; j += 2) {
                        const float2 vl = make_float2(lo[j], lo[j + 1]), vh = make_float2(hi[j], hi[j + 1]);
                        *reinterpret_cast<float2*>(orow + (2 * p) * ROWS + j) = vl;
                        *reinterpret_cast<float2*>(orow + (2 * p + 1) * ROWS + j) = vh;
                        *reinterpret_cast<float2*>(ocK + (2 * p) * ROWS + j) = vl;
                        *reinterpret_cast<float2*>(ocK + (2 * p + 1) * ROWS + j) = vh;
                    }
                }
            }
        }
        __syncthreads();   // s_act = a_L

        // ---- output layer (k_mlp_deep's arithmetic: pairs from the parameter block, h ascending) and y_bar --------
        {
            constexpr int PASSES = (NROW + NT - 1) / NT;
            const float4 b2 = w.b2;
#pragma unroll
            for (int pass = 0; pass < PASSES; ++pass) {
                const int r_raw = threadIdx.x + NT * pass;
                const int r = r_raw < NROW ? r_raw : NROW - 1;   // idle threads of the last pass redo a row: convergent
                const int rbk = r / ROWS, row = r - rbk * ROWS;  // loop, W2 by uniform loads; they store nothing
                const float* src = s_act + (rbk * H) * ROWS + row;
                f32x2 q01 = pack2(b2.x, b2.y), q23 = pack2(b2.z, b2.w);
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    const float4 cw = w.w2[h];   // {W2[1,h], W2[0,h], W2[3,h], W2[2,h]}
                    const f32x2 aa = bcast2(src[h * ROWS]);
                    q01 = add2_rn_swapped(q01, mul2_rn(aa, pack2(cw.x, cw.y)));
                    q23 = add2_rn_swapped(q23, mul2_rn(aa, pack2(cw.z, cw.w)));
                }
                float y[4];
                unpack2(q01, y[0], y[1]);
                unpack2(q23, y[2], y[3]);
                const long long p = tile * PTS_TILE + r;
                if (r_raw < NROW) {
                    float4 yb = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (p < n) {
                        const float4 t4 = __ldg(a.target + p);
                        const float tg[4] = {t4.x, t4.y, t4.z, t4.w};
                        float d[4];
#pragma unroll
                        for (int o = 0; o < 4; ++o) {
                            const double e = double(y[o]) - double(tg[o]);
                            red[4] += a.lam[o] * (e * e);
                            d[o] = __fmul_rn(a.coef[o], __fsub_rn(y[o], tg[o]));
                        }
                        yb = make_float4(d[0], d[1], d[2], d[3]);
                        red[0] += double(yb.x); red[1] += double(yb.y); red[2] += double(yb.z); red[3] += double(yb.w);
                    }
                    s_row[r] = yb;
                }
            }
        }
        __syncthreads();

        // ================= backward (k_deep_grad's) ======================================================================
        // ---- output layer: dW2[o,h] = sum_rows y_bar_o a_L[h]  (warp per unit, lanes over rows) -------------------
        for (int h = warp; h < H; h += NT / 32) {
            float d[4] = {0.f, 0.f, 0.f, 0.f};
            for (int r = lane; r < NROW; r += 32) {
                const int rbk = r / ROWS, row = r - rbk * ROWS;
                const float av = s_act[(rbk * H + h) * ROWS + row];
                const float4 yb = s_row[r];
                d[0] = __fmaf_rn(yb.x, av, d[0]); d[1] = __fmaf_rn(yb.y, av, d[1]);
                d[2] = __fmaf_rn(yb.z, av, d[2]); d[3] = __fmaf_rn(yb.w, av, d[3]);
            }
#pragma unroll
            for (int o = 0; o < 4; ++o) {
                const float v = warp_sum_f(d[o]);
                if (lane == 0) part[oW2 + size_t(o) * H + h] += double(v);
            }
        }
        __syncthreads();
        // ---- delta_a_L = W2^T y_bar, in place ---------------------------------------------------------------------
        for (int i = threadIdx.x; i < ACT; i += NT) {
            const int row = i % ROWS, hb = i / ROWS, h = hb % H, rbk = hb / H;
            const float4 yb = s_row[rbk * ROWS + row];
            const float w0 = __ldg(a.W2 + h), w1 = __ldg(a.W2 + H + h), w2 = __ldg(a.W2 + 2 * H + h), w3 = __ldg(a.W2 + 3 * H + h);
            s_act[i] = __fmaf_rn(w3, yb.w, __fmaf_rn(w2, yb.z, __fmaf_rn(w1, yb.y, w0 * yb.x)));
        }
        // ---- hidden layers, last to first ---------------------------------------------------------------------------
        for (int k = nl - 1; k >= 0; --k) {
            __syncthreads();   // delta_a_{k+2} is complete in s_act
            // mask: delta_z = delta_a (.) (a_{k+2} > 0)
            {
                const float4* ak = reinterpret_cast<const float4*>(ck + size_t(k + 1) * ACT);
                float4* d4 = reinterpret_cast<float4*>(s_act);
                for (int i = threadIdx.x; i < ACT / 4; i += NT) {
                    const float4 m = ak[i];
                    float4 v = d4[i];
                    v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f;
                    v.z = m.z > 0.f ? v.z : 0.f; v.w = m.w > 0.f ? v.w : 0.f;
                    d4[i] = v;
                }
            }
            // dWh[k][g][h] += sum_rows delta_z[g] a_{k+1}[h],  dbh[k][g] += sum_rows delta_z[g]:
            // warp w owns g in [w GW, (w+1) GW), lane owns h = lane + 32 j; a_{k+1} staged transposed [r][H+1]
            {
                constexpr int GW = H / 8, HJ = H / 32;
                const int gw0 = warp * GW;
                float acc[GW][HJ], sb[GW];
#pragma unroll
                for (int gg = 0; gg < GW; ++gg) {
                    sb[gg] = 0.f;
#pragma unroll
                    for (int j = 0; j < HJ; ++j) acc[gg][j] = 0.f;
                }
                const float* aprev = ck + size_t(k) * ACT;
                for (int rbk = 0; rbk < RB; ++rbk)
                    for (int r0 = 0; r0 < ROWS; r0 += CH) {
                        __syncthreads();   // the mask is applied / the previous chunk has been read
                        for (int i = threadIdx.x; i < H * CH; i += NT) {
                            const int h = i / CH, r = i - h * CH;
                            s_scr[r * (H + 1) + h] = aprev[(rbk * H + h) * ROWS + r0 + r];
                        }
                        __syncthreads();
                        const float* dz = s_act + (rbk * H + gw0) * ROWS + r0;
#pragma unroll 2
                        for (int r = 0; r < CH; r += 2) {
                            float2 dv[GW];
                            float av[2][HJ];
#pragma unroll
                            for (int gg = 0; gg < GW; ++gg) dv[gg] = *reinterpret_cast<const float2*>(dz + gg * ROWS + r);
#pragma unroll
                            for (int j = 0; j < HJ; ++j) {
                                av[0][j] = s_scr[r * (H + 1) + lane + 32 * j];
                                av[1][j] = s_scr[(r + 1) * (H + 1) + lane + 32 * j];
                            }
#pragma unroll
                            for (int gg = 0; gg < GW; ++gg) {
                                sb[gg] += dv[gg].x + dv[gg].y;
#pragma unroll
                                for (int j = 0; j < HJ; ++j) acc[gg][j] = __fmaf_rn(dv[gg].y, av[1][j], __fmaf_rn(dv[gg].x, av[0][j], acc[gg][j]));
                            }
                        }
                    }
                double* pw = part + oWh + size_t(k) * H * H;
#pragma unroll
                for (int gg = 0; gg < GW; ++gg) {
#pragma unroll
                    for (int j = 0; j < HJ; ++j) pw[size_t(gw0 + gg) * H + lane + 32 * j] += double(acc[gg][j]);
                    if (lane == 0) part[obh + size_t(k) * H + gw0 + gg] += double(sb[gg]);
                }
            }
            cp_async_wait_all();
            __syncthreads();   // layer k's weights have landed; every warp is done with the staging area
            // delta_a_{k+1}[h] = sum_g W[g,h] delta_z[g]: warp = 16 outputs h of its row-block, lane = 6 rows;
            // s_w[h H + g] holds the pair {W[g+1,h], W[g,h]} for even g
            {
                float acc[PT][GT];
#pragma unroll
                for (int j = 0; j < PT; ++j)
#pragma unroll
                    for (int hh = 0; hh < GT; ++hh) acc[j][hh] = 0.f;
                const float* drow = s_act + (rb * H) * ROWS + lane * PT;
#pragma unroll 2
                for (int g = 0; g < H; g += 2) {
                    float d0[PT], d1[PT];
#pragma unroll
                    for (int j = 0; j < PT; j += 2) {
                        const float2 t0 = *reinterpret_cast<const float2*>(drow + g * ROWS + j);
                        const float2 t1 = *reinterpret_cast<const float2*>(drow + (g + 1) * ROWS + j);
                        d0[j] = t0.x; d0[j + 1] = t0.y; d1[j] = t1.x; d1[j + 1] = t1.y;
                    }
#pragma unroll
                    for (int hh = 0; hh < GT; ++hh) {
                        const float2 wp = *reinterpret_cast<const float2*>(s_w + (g0 + hh) * H + g);   // {W[g+1,h], W[g,h]}
#pragma unroll
                        for (int j = 0; j < PT; ++j) acc[j][hh] = __fmaf_rn(wp.x, d1[j], __fmaf_rn(wp.y, d0[j], acc[j][hh]));
                    }
                }
                __syncthreads();   // every warp has read delta_z and the weights
                if (k > 0) load_layer(k - 1);
                float* orow = s_act + (rb * H + g0) * ROWS + lane * PT;
#pragma unroll
                for (int hh = 0; hh < GT; ++hh)
#pragma unroll
                    for (int j = 0; j < PT; j += 2)
                        *reinterpret_cast<float2*>(orow + hh * ROWS + j) = make_float2(acc[j][hh], acc[j + 1][hh]);
            }
        }
        __syncthreads();   // delta_a_1 complete
        // ---- layer 1: delta_z_1 = delta_a_1 (.) (a_1 > 0); dW1[h,:] += sum delta_z_1 (x, y, z, t), db1 += sum delta_z_1
        {
            const float4* a1 = reinterpret_cast<const float4*>(ck);
            float4* d4 = reinterpret_cast<float4*>(s_act);
            for (int i = threadIdx.x; i < ACT / 4; i += NT) {
                const float4 m = a1[i];
                float4 v = d4[i];
                v.x = m.x > 0.f ? v.x : 0.f; v.y = m.y > 0.f ? v.y : 0.f;
                v.z = m.z > 0.f ? v.z : 0.f; v.w = m.w > 0.f ? v.w : 0.f;
                d4[i] = v;
            }
            for (int r = threadIdx.x; r < NROW; r += NT) {
                long long p = tile * PTS_TILE + r;
                if (p > n - 1) p = n - 1;
                s_row[r] = __ldg(a.x + p);
            }
        }
        __syncthreads();
        for (int h = warp; h < H; h += NT / 32) {
            float d[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
            for (int r = lane; r < NROW; r += 32) {
                const int rbk = r / ROWS, row = r - rbk * ROWS;
                const float dz = s_act[(rbk * H + h) * ROWS + row];
                const float4 c = s_row[r];
                d[0] = __fmaf_rn(dz, c.x, d[0]); d[1] = __fmaf_rn(dz, c.y, d[1]);
                d[2] = __fmaf_rn(dz, c.z, d[2]); d[3] = __fmaf_rn(dz, c.w, d[3]);
                d[4] += dz;
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float v = warp_sum_f(d[kk]);
                if (lane == 0) part[oW1 + size_t(h) * 4 + kk] += double(v);
            }
            const float v = warp_sum_f(d[4]);
            if (lane == 0) part[ob1 + h] += double(v);
        }
        __syncthreads();   // the next tile's layer 1 overwrites s_act and s_row
    }
    cp_async_wait_all();
    // db2 and the loss sum: warps in order, then the block's slots
#pragma unroll
    for (int o = 0; o < 5; ++o) {
        const double v = warp_sum_d(red[o]);
        if (lane == 0) s_red[warp][o] = v;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        double s = 0.0;
        for (int w8 = 0; w8 < NT / 32; ++w8) s += s_red[w8][threadIdx.x];
        part[threadIdx.x < 4 ? ob2 + threadIdx.x : P] = s;
    }
}

// one thread per entry: block partials summed in block order
__global__ void k_deep_data_reduce(const double* __restrict__ partials, int blocks, size_t P, double* grad, double* acc) {
    const size_t e = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= P + 1) return;
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += partials[size_t(b) * (P + 1) + e];
    if (e < P) grad[e] = s;
    else acc[0] = s;
}

template <int H>
int launch_t(const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    constexpr size_t smem = Geo<H>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_deep_data_grad<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_deep_data_grad<H><<<blocks, NT, smem, st>>>(*static_cast<const MlpConst<H>*>(mlp_const), a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    const size_t P = grad_len(H, a.hidden_layers);
    k_deep_data_reduce<<<unsigned((P + 1 + 255) / 256), 256, 0, st>>>(a.partials, blocks, P, grad, acc);
    return int(cudaGetLastError());
}

}  // namespace

size_t deep_data_ckpt_floats(int H, int hidden_layers) {
    (void)H;   // RB x H x ROWS = 8 x 16 x 192 for every width
    return size_t(hidden_layers) * Geo<32>::ACT;
}

int deep_data_blocks(int H, long long n_points, int max_blocks) {
    const int pts = H == 32 ? Geo<32>::NROW : (H == 64 ? Geo<64>::NROW : Geo<128>::NROW);
    const long long tiles = (n_points + pts - 1) / pts;
    return int(tiles < max_blocks ? (tiles > 0 ? tiles : 1) : max_blocks);
}

int deep_data_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    switch (H) {
        case 32: return launch_t<32>(mlp_const, a, blocks, grad, acc, st);
        case 64: return launch_t<64>(mlp_const, a, blocks, grad, acc, st);
        case 128: return launch_t<128>(mlp_const, a, blocks, grad, acc, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
