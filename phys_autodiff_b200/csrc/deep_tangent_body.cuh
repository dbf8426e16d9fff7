// The kernel behind k_deep_tangent (deep_tangent_kernels.cu) and k_colloc_tangent (colloc_tangent_kernels.cu); see
// deep_tangent_kernels.cuh for what they compute.  The two differ only in where a point's inputs come from.  Each of the
// two files includes this one once, after defining
//   DEEP_TANGENT_KERNEL   the kernel's name;
//   DEEP_TANGENT_POINTS   its row source: false, the slab's grid points in linear order (coordinates from the axis tables,
//                         one time input a.tc); true, the caller's points a.pts[0 .. a.n_points) (one float4 per point,
//                         its own time input).
// The body is the kernel itself, not a __device__ function both kernels inline: inlined, it loses the thread-index range
// that __launch_bounds__ gives the kernel, and k_deep_tangent<128, *> compiles to different code.
//
// Both use k_deep_grad's tile geometry (256 threads, a warp owns 16 units of one row-block) with 5 rows per point
// instead of 3 slices: a lane holds the 5 rows of ONE point (value row j = 0, tangent rows j = 1 + k), so a row-block
// has 160 rows and act[row-block][h][160] is 80 KB for every H (H = 128: 1 row-block, 64: 2, 32: 4).
// One point per lane rather than two keeps the 5 rows a lane owns contiguous; the price is scalar LDS for the row
// operands (an odd row count per lane rules out LDS.64), which the weight broadcasts and 80 math instructions per input
// unit absorb.  Per hidden layer a warp keeps 8 packed value accumulators (16 units, FMUL2 / FADD2 un-contracted by the
// half-swap trick, k_mlp_deep's order) and 4 x 16 scalar tangent accumulators (FFMA): 1 strict row + 4 FMA rows =
// about three strict-row equivalents of FP32-pipe time per point, the same as the strict fields pass's three slices.
// Per tile:
//   forward   layer 1, hidden layers (outputs in place, weights staged one layer at a time through one shared buffer
//             with cp.async), output layer (a thread per (output, point)), residuals (a thread per point).
//   GRAD      every layer's 5-row activations also go to the block's checkpoint area (global memory, L x 80 KB per block,
//             meant to stay in L2).  Seeds of DESIGN section 4.6.1 per row: value row y_bar, tangent row k the column
//             J_bar[:,k].  Then k_deep_grad's backward with the rules of the tangent rows: every row masked by its
//             point's VALUE mask, dbh and db1 from the value rows only, dW1[h,k] += delta_value[h] c_k + delta_tan,k[h].
// No FFMA2 and no tcgen05: the value row keeps k_mlp_deep's FMUL2 / FADD2, everything else is scalar FFMA.
#if !defined(DEEP_TANGENT_KERNEL) || !defined(DEEP_TANGENT_POINTS)
#error "define DEEP_TANGENT_KERNEL and DEEP_TANGENT_POINTS before including deep_tangent_body.cuh"
#endif
#include "deep_tangent_kernels.cuh"
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

constexpr int NT = DEEP_TANGENT_THREADS;
constexpr int GT = 16;          // units per warp
constexpr int PT = 5;           // rows per lane: value, d/dc_x, d/dc_y, d/dc_z, d/dc_t of one point
constexpr int ROWS = 32 * PT;   // rows per row-block
constexpr int CH = 8 * PT;      // rows per staging chunk of the dW step (whole points)
constexpr int NOUT = 4 * PT;    // y_o and J[o][0..3] of one point

constexpr int cmax(int x, int y) { return x > y ? x : y; }

template <int H, bool GRAD>
struct Geo {
    static constexpr int G = H / GT;               // warps per row-block
    static constexpr int RB = 8 / G;               // row-blocks per tile
    static constexpr int NROW = RB * ROWS;         // rows per tile
    static constexpr int PTS_TILE = RB * 32;       // points per tile
    static constexpr int ACT = RB * H * ROWS;      // floats of one layer's activations (20480 for every H)
    // outputs [PTS_TILE][20] | per-row seeds / coordinates [NROW] float4 (the same 20 floats per point) | dW staging
    static constexpr int SCR = GRAD ? cmax(CH * (H + 1), NOUT * PTS_TILE) : NOUT * PTS_TILE;
    static constexpr size_t SMEM = (size_t(ACT) + 5 * H + H * H + SCR) * sizeof(float);
};

__host__ __device__ constexpr size_t grad_len(int H, int L) {
    return size_t(9) * H + 4 + size_t(L - 1) * (size_t(H) * H + H);
}

template <int H, bool GRAD>
__global__ void __launch_bounds__(NT, 1) DEEP_TANGENT_KERNEL(const __grid_constant__ DeepTangentArgs a) {
    constexpr bool POINTS = DEEP_TANGENT_POINTS;
    using Q = Geo<H, GRAD>;
    constexpr int G = Q::G, RB = Q::RB, NROW = Q::NROW, PTS_TILE = Q::PTS_TILE, ACT = Q::ACT;
    extern __shared__ __align__(16) float smem[];
    float* s_act = smem;                                              // [RB][H][ROWS]
    float2* s_l1 = reinterpret_cast<float2*>(smem + ACT);             // [5][H/2] layer-1 pairs (as k_mlp_deep)
    float* s_w = smem + ACT + 5 * H;                                  // [H][H] one hidden layer, k_mlp_deep's layout
    float* s_scr = s_w + H * H;
    float* s_out = s_scr;                                             // [PTS_TILE][o][y | J[o][0..3]]
    float4* s_row = reinterpret_cast<float4*>(s_scr);                 // [NROW] seeds, later layer-1 coefficients
    __shared__ double s_red[NT / 32][6];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rb = warp / G, g0 = (warp % G) * GT;
    const int L = a.hidden_layers, nl = L - 1;
    const long long n_slab = POINTS ? a.n_points : (long long)(a.z_end - a.z_begin) * a.ny * a.nx;
    const long long tiles = (n_slab + PTS_TILE - 1) / PTS_TILE;
    const int plane = a.nx * a.ny;

    const size_t P = GRAD ? grad_len(H, L) : 0;
    const size_t oW1 = 0, ob1 = 4 * H, oWh = 5 * H, obh = oWh + size_t(nl) * H * H, oW2 = obh + size_t(nl) * H, ob2 = oW2 + 4 * H;
    double* part = a.partials + size_t(blockIdx.x) * (P + 2);
    float* ck = GRAD ? a.ckpt + size_t(blockIdx.x) * L * ACT : nullptr;
    if (GRAD)
        for (size_t e = threadIdx.x; e < P + 2; e += NT) part[e] = 0.0;

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
    double red[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};   // db2[4], sum R_sigma^2, sum |R_u|^2
    __syncthreads();

    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        if (nl > 0 && wcur != 0) load_layer(0);   // s_w is free: the previous tile's last reader is behind a barrier
        // ================= forward ================================================================================
        // ---- layer 1: value row with k_mlp_deep's arithmetic at slice t; tangent rows m (.) W1[:,k] ----------------
        {
            long long p = tile * PTS_TILE + rb * 32 + lane;
            if (p > n_slab - 1) p = n_slab - 1;   // tail tile: a valid point, its seeds are zero and it is not summed
            float cx, cy, cz, ct;
            if (POINTS) {
                const float4 c4 = __ldg(a.pts + p);
                cx = c4.x; cy = c4.y; cz = c4.z; ct = c4.w;
            } else {
                const int zl = int(p / plane), rem = int(p - (long long)zl * plane);
                const int y = rem / a.nx, x = rem - y * a.nx;
                cx = __ldg(a.cxs + x); cy = __ldg(a.cys + y); cz = __ldg(a.czs + a.z_begin + zl); ct = a.tc;
            }
            const int off = (rb * H) * ROWS + lane * PT;
            float* dst = s_act + off;
#pragma unroll 2
            for (int q = 0; q < GT / 2; ++q) {
                const int qq = g0 / 2 + q;
                const float2 b1p = s_l1[qq], w0s = s_l1[H / 2 + qq], w1s = s_l1[2 * (H / 2) + qq], w2s = s_l1[3 * (H / 2) + qq];
                const float2 w3 = s_l1[4 * (H / 2) + qq];
                const float2 t0 = make_float2(__fmul_rn(w3.x, ct), __fmul_rn(w3.y, ct));   // the IEEE product, per row
                const f32x2 sx = add2_rn_swapped(pack2(b1p), mul2_rn(pack2(w0s), bcast2(cx)));
                const f32x2 sxy = add2_rn_swapped(sx, mul2_rn(pack2(w1s), bcast2(cy)));
                const f32x2 sxyz = add2_rn_swapped(sxy, mul2_rn(pack2(w2s), bcast2(cz)));
                float z0, z1;
                unpack2(add2_rn(sxyz, pack2(t0)), z0, z1);
                const bool m0 = z0 > 0.f, m1 = z1 > 0.f;
                // unit 2qq: W1[., 0..3] = w0s.y, w1s.y, w2s.y, w3.x;  unit 2qq+1: w0s.x, w1s.x, w2s.x, w3.y
                const float v0[PT] = {relu_ref(z0), m0 ? w0s.y : 0.f, m0 ? w1s.y : 0.f, m0 ? w2s.y : 0.f, m0 ? w3.x : 0.f};
                const float v1[PT] = {relu_ref(z1), m1 ? w0s.x : 0.f, m1 ? w1s.x : 0.f, m1 ? w2s.x : 0.f, m1 ? w3.y : 0.f};
#pragma unroll
                for (int j = 0; j < PT; ++j) {
                    dst[(2 * qq) * ROWS + j] = v0[j];
                    dst[(2 * qq + 1) * ROWS + j] = v1[j];
                    if (GRAD) {
                        ck[off + (2 * qq) * ROWS + j] = v0[j];
                        ck[off + (2 * qq + 1) * ROWS + j] = v1[j];
                    }
                }
            }
        }
        // ---- hidden -> hidden layers ------------------------------------------------------------------------------
        for (int l = 0; l < nl; ++l) {
            cp_async_wait_all();
            __syncthreads();   // layer l's weights have landed, its inputs are written
            const float* wbuf = s_w + g0;
            const float* arow = s_act + (rb * H) * ROWS + lane * PT;
            f32x2 qv[GT / 2];   // value row, unit pairs (g0 + 2p, g0 + 2p + 1)
            float qt[4][GT];    // tangent rows
            {
                const float* bl = a.bh + size_t(l) * H + g0;
#pragma unroll
                for (int p = 0; p < GT / 2; ++p) {
                    const float2 b = __ldg(reinterpret_cast<const float2*>(bl) + p);
                    qv[p] = pack2(b.x, b.y);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int gg = 0; gg < GT; ++gg) qt[k][gg] = 0.f;
            }
#pragma unroll 2
            for (int h = 0; h < H; ++h) {
                float av[PT];
                float4 wv[GT / 4];
#pragma unroll
                for (int j = 0; j < PT; ++j) av[j] = arow[h * ROWS + j];
#pragma unroll
                for (int v = 0; v < GT / 4; ++v) wv[v] = *reinterpret_cast<const float4*>(wbuf + h * H + 4 * v);
                const f32x2 aa = bcast2(av[0]);
#pragma unroll
                for (int v = 0; v < GT / 4; ++v) {   // {W[g+1,h], W[g,h], W[g+3,h], W[g+2,h]}
                    qv[2 * v] = add2_rn_swapped(qv[2 * v], mul2_rn(aa, pack2(wv[v].x, wv[v].y)));
                    qv[2 * v + 1] = add2_rn_swapped(qv[2 * v + 1], mul2_rn(aa, pack2(wv[v].z, wv[v].w)));
                }
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int v = 0; v < GT / 4; ++v) {
                        qt[k][4 * v] = __fmaf_rn(wv[v].y, av[1 + k], qt[k][4 * v]);
                        qt[k][4 * v + 1] = __fmaf_rn(wv[v].x, av[1 + k], qt[k][4 * v + 1]);
                        qt[k][4 * v + 2] = __fmaf_rn(wv[v].w, av[1 + k], qt[k][4 * v + 2]);
                        qt[k][4 * v + 3] = __fmaf_rn(wv[v].z, av[1 + k], qt[k][4 * v + 3]);
                    }
            }
            __syncthreads();   // every warp has read this layer's inputs and weights
            if (GRAD) {
                if (l + 1 < nl) load_layer(l + 1);   // the last forward layer's weights are the first backward layer's
            } else if (nl > 1) {
                load_layer(l + 1 < nl ? l + 1 : 0);  // the next layer's, or the next tile's first
            }
            {
                const int off = (rb * H + g0) * ROWS + lane * PT;
                float* orow = s_act + off;
#pragma unroll
                for (int p = 0; p < GT / 2; ++p) {
                    float zz[2];
                    unpack2(qv[p], zz[0], zz[1]);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int gg = 2 * p + e;
                        const bool m = zz[e] > 0.f;
                        const float v[PT] = {relu_ref(zz[e]), m ? qt[0][gg] : 0.f, m ? qt[1][gg] : 0.f, m ? qt[2][gg] : 0.f,
                                             m ? qt[3][gg] : 0.f};
#pragma unroll
                        for (int j = 0; j < PT; ++j) {
                            orow[gg * ROWS + j] = v[j];
                            if (GRAD) ck[size_t(l + 1) * ACT + off + gg * ROWS + j] = v[j];
                        }
                    }
                }
            }
        }
        __syncthreads();   // s_act = a_L (5 rows per point)
        // ---- output layer: y_o strict (k_mlp_deep's order), J[o][k] with FFMA from +0, h ascending ------------------
        for (int i = threadIdx.x; i < 4 * PTS_TILE; i += NT) {
            const int o = i / PTS_TILE, pt = i - o * PTS_TILE;   // o is warp-uniform: W2 arrives by broadcast loads
            const float* src = s_act + ((pt / 32) * H) * ROWS + (pt % 32) * PT;
            const float* w2 = a.W2 + size_t(o) * H;
            float yo = __ldg(a.b2 + o), J[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
            for (int h = 0; h < H; ++h) {
                const float w = __ldg(w2 + h);
                yo = __fadd_rn(yo, __fmul_rn(w, src[h * ROWS]));
#pragma unroll
                for (int k = 0; k < 4; ++k) J[k] = __fmaf_rn(w, src[h * ROWS + 1 + k], J[k]);
            }
            float* d = s_out + pt * NOUT + o * PT;
            d[0] = yo; d[1] = J[0]; d[2] = J[1]; d[3] = J[2]; d[4] = J[3];
        }
        __syncthreads();
        // ---- residuals (k_tangent_loss's arithmetic), the two sums and, for GRAD, the per-row seeds -----------------
        for (int pt = threadIdx.x; pt < PTS_TILE; pt += NT) {
            const long long p = tile * PTS_TILE + pt;
            float y[4], J[4][4];
#pragma unroll
            for (int o = 0; o < 4; ++o) {
                y[o] = s_out[pt * NOUT + o * PT];
#pragma unroll
                for (int k = 0; k < 4; ++k) J[o][k] = s_out[pt * NOUT + o * PT + 1 + k];
            }
            float4 seed[PT];
#pragma unroll
            for (int j = 0; j < PT; ++j) seed[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p < n_slab) {
                const float s[3] = {a.sx, a.sy, a.sz};
                float g[4][3];   // d y_o / d x_j
#pragma unroll
                for (int o = 0; o < 4; ++o)
#pragma unroll
                    for (int j = 0; j < 3; ++j) g[o][j] = J[o][j] * s[j];
                const float div = (g[1][0] + g[2][1]) + g[3][2];
                float R[4];
#pragma unroll
                for (int o = 0; o < 4; ++o) R[o] = J[o][3] + ((y[1] * g[o][0] + y[2] * g[o][1]) + y[3] * g[o][2]);
                R[0] += y[0] * div;
                red[4] += double(R[0]) * double(R[0]);
                red[5] += double(R[1]) * double(R[1]) + double(R[2]) * double(R[2]) + double(R[3]) * double(R[3]);
                if (!GRAD && POINTS && a.R_pts) a.R_pts[p] = make_float4(R[0], R[1], R[2], R[3]);
                if (!GRAD && !POINTS && a.R[0]) {
                    a.R[0][p] = R[0]; a.R[1][p] = R[1]; a.R[2][p] = R[2]; a.R[3][p] = R[3];
                }
                if (GRAD) {
                    // DESIGN section 4.6.1: g_o = (2 w_o / N) R_o;  y_bar_0 = g_0 div,  y_bar_{j+1} = sum_o g_o s_j J[o][j];
                    // J_bar[o][3] = g_o,  J_bar[o][j] = s_j (g_o y_{j+1} + [o = j+1] g_0 y_0)
                    const float gb[4] = {a.scale_s * R[0], a.scale_u * R[1], a.scale_u * R[2], a.scale_u * R[3]};
                    float yb[4], Jb[4][4];
                    yb[0] = gb[0] * div;
#pragma unroll
                    for (int j = 0; j < 3; ++j) yb[j + 1] = ((gb[0] * g[0][j] + gb[1] * g[1][j]) + gb[2] * g[2][j]) + gb[3] * g[3][j];
#pragma unroll
                    for (int o = 0; o < 4; ++o) {
                        Jb[o][3] = gb[o];
#pragma unroll
                        for (int j = 0; j < 3; ++j) Jb[o][j] = s[j] * (gb[o] * y[j + 1] + (o == j + 1 ? gb[0] * y[0] : 0.f));
                    }
                    seed[0] = make_float4(yb[0], yb[1], yb[2], yb[3]);
#pragma unroll
                    for (int k = 0; k < 4; ++k) seed[1 + k] = make_float4(Jb[0][k], Jb[1][k], Jb[2][k], Jb[3][k]);
                    red[0] += double(yb[0]); red[1] += double(yb[1]); red[2] += double(yb[2]); red[3] += double(yb[3]);
                }
            }
            if (GRAD) {
                // the point's 5 rows are rows pt * 5 .. pt * 5 + 4 of the tile: the same 20 floats it has just read
#pragma unroll
                for (int j = 0; j < PT; ++j) s_row[pt * PT + j] = seed[j];
            }
        }
        if (!GRAD) {
            __syncthreads();   // the next tile's output stage overwrites s_out, its layer 1 s_act
            continue;
        }
        __syncthreads();

        // ================= backward (GRAD) =========================================================================
        // ---- output layer: dW2[o,h] = sum_rows seed_o a_L[h]  (warp per unit, lanes over rows) ---------------------
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
        // ---- row adjoints W2^T seed, in place -----------------------------------------------------------------------
        for (int i = threadIdx.x; i < ACT; i += NT) {
            const int row = i % ROWS, hb = i / ROWS, h = hb % H, rbk = hb / H;
            const float4 yb = s_row[rbk * ROWS + row];
            const float w0 = __ldg(a.W2 + h), w1 = __ldg(a.W2 + H + h), w2 = __ldg(a.W2 + 2 * H + h), w3 = __ldg(a.W2 + 3 * H + h);
            s_act[i] = __fmaf_rn(w3, yb.w, __fmaf_rn(w2, yb.z, __fmaf_rn(w1, yb.y, w0 * yb.x)));
        }
        // every row of a point masked by the point's value-row activation of checkpoint layer `layer`
        auto mask_rows = [&](int layer) {
            const float* ak = ck + size_t(layer) * ACT;
            for (int i = threadIdx.x; i < ACT / PT; i += NT) {   // (row-block, unit, point); consecutive threads: points
                const int b = i * PT;
                if (!(ak[b] > 0.f)) {
#pragma unroll
                    for (int j = 0; j < PT; ++j) s_act[b + j] = 0.f;
                }
            }
        };
        // ---- hidden layers, last to first ---------------------------------------------------------------------------
        for (int k = nl - 1; k >= 0; --k) {
            __syncthreads();   // the adjoint of layer k+2's activations is complete in s_act
            mask_rows(k + 1);
            // dWh[k][g][h] += sum_rows delta[g] a_{k+1}[h]  (every row),  dbh[k][g] += sum_{value rows} delta[g]:
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
                        for (int r = 0; r < CH; r += PT) {
#pragma unroll
                            for (int j = 0; j < PT; ++j) {
                                float dv[GW], av[HJ];
#pragma unroll
                                for (int gg = 0; gg < GW; ++gg) dv[gg] = dz[gg * ROWS + r + j];
#pragma unroll
                                for (int jj = 0; jj < HJ; ++jj) av[jj] = s_scr[(r + j) * (H + 1) + lane + 32 * jj];
#pragma unroll
                                for (int gg = 0; gg < GW; ++gg) {
                                    if (j == 0) sb[gg] += dv[gg];
#pragma unroll
                                    for (int jj = 0; jj < HJ; ++jj) acc[gg][jj] = __fmaf_rn(dv[gg], av[jj], acc[gg][jj]);
                                }
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
            // adjoint of a_{k+1}[h] = sum_g W[g,h] delta[g]: warp = 16 units h of its row-block, lane = its point's 5 rows;
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
                    for (int j = 0; j < PT; ++j) {
                        d0[j] = drow[g * ROWS + j];
                        d1[j] = drow[(g + 1) * ROWS + j];
                    }
#pragma unroll
                    for (int hh = 0; hh < GT; ++hh) {
                        const float2 wp = *reinterpret_cast<const float2*>(s_w + (g0 + hh) * H + g);   // {W[g+1,h], W[g,h]}
#pragma unroll
                        for (int j = 0; j < PT; ++j) acc[j][hh] = __fmaf_rn(wp.x, d1[j], __fmaf_rn(wp.y, d0[j], acc[j][hh]));
                    }
                }
                __syncthreads();   // every warp has read the deltas and the weights
                if (k > 0) load_layer(k - 1);
                float* orow = s_act + (rb * H + g0) * ROWS + lane * PT;
#pragma unroll
                for (int hh = 0; hh < GT; ++hh)
#pragma unroll
                    for (int j = 0; j < PT; ++j) orow[hh * ROWS + j] = acc[j][hh];
            }
        }
        __syncthreads();   // the adjoint of a_1 is complete
        // ---- layer 1: delta_1 = adjoint (.) m_1; dW1[h,k] += delta_value c_k + delta_tan,k, db1 += delta_value --------
        mask_rows(0);
        for (int r = threadIdx.x; r < NROW; r += NT) {
            const int pt = r / PT, j = r - pt * PT;
            float4 cf;
            if (j == 0) {
                long long p = tile * PTS_TILE + pt;
                if (p > n_slab - 1) p = n_slab - 1;
                if (POINTS) {
                    cf = __ldg(a.pts + p);
                } else {
                    const int zl = int(p / plane), rem = int(p - (long long)zl * plane);
                    const int y = rem / a.nx, x = rem - y * a.nx;
                    cf = make_float4(__ldg(a.cxs + x), __ldg(a.cys + y), __ldg(a.czs + a.z_begin + zl), a.tc);
                }
            } else {
                cf = make_float4(j == 1 ? 1.f : 0.f, j == 2 ? 1.f : 0.f, j == 3 ? 1.f : 0.f, j == 4 ? 1.f : 0.f);
            }
            s_row[r] = cf;   // tile row r = point r / 5, row r % 5 (row-block r / ROWS: ROWS is a multiple of 5)
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
                if (row % PT == 0) d[4] += dz;
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float v = warp_sum_f(d[kk]);
                if (lane == 0) part[oW1 + size_t(h) * 4 + kk] += double(v);
            }
            const float v = warp_sum_f(d[4]);
            if (lane == 0) part[ob1 + h] += double(v);
        }
        __syncthreads();   // the next tile's layer 1 overwrites s_act and its output stage s_row
    }
    cp_async_wait_all();
    // db2 and the two residual sums: warps in order, then the block's slots
#pragma unroll
    for (int o = 0; o < 6; ++o) {
        const double v = warp_sum_d(red[o]);
        if (lane == 0) s_red[warp][o] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6 && (GRAD || threadIdx.x >= 4)) {
        double s = 0.0;
        for (int w = 0; w < NT / 32; ++w) s += s_red[w][threadIdx.x];
        part[threadIdx.x < 4 ? ob2 + threadIdx.x : P + (threadIdx.x - 4)] = s;
    }
}

}  // namespace

}  // namespace physad
