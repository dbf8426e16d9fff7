// The deep closed-loop kernels; see deep_grad_kernels.cuh for what they compute.
//
// k_deep_grad<H> uses k_mlp_deep's tile geometry (256 threads, a warp owns 16 units of one row-block, a lane 6 rows =
// 2 points x 3 slices; H = 128: 1 row-block of 192 rows, 64: 2, 32: 4) and its shared-memory activation buffer
// act[row-block][h][192].  Per tile:
//   forward   layer 1 and the hidden layers with k_mlp_deep's code (same roundings in the same order: bit-identical
//             pre-activations, hence the same ReLU masks), every layer's activations also stored to the block's
//             checkpoint area (global memory; L x 96 KB per block, meant to stay in L2).  The output layer is not needed.
//   backward  y_bar of every row -> dW2, db2 and delta_a_L = W2^T y_bar (in place in act); then for every hidden layer,
//             last to first: delta_z = delta_a (.) (a > 0)  [mask from the checkpoint], dWh += delta_z a_prev^T and
//             dbh += sum delta_z  [a_prev staged transposed from the checkpoint, 64 rows at a time],
//             delta_a_prev = W^T delta_z  [register-tiled like the forward, outputs written in place after a barrier];
//             finally delta_z_1 -> dW1 (against the row's coordinates) and db1.
// The hidden->hidden weights are staged one layer at a time in one shared buffer (cp.async, issued as soon as the
// previous contraction has read the buffer, so the copy overlaps the element-wise and dW work); the second buffer of
// k_mlp_deep's layout is the staging area of the dW step and of the per-row y_bar / coordinates.
// No FFMA2 anywhere: the forward keeps k_mlp_deep's un-contracted FMUL2 / FADD2, the backward uses scalar FFMA.
#include "deep_grad_kernels.cuh"
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

constexpr int NT = DEEP_GRAD_THREADS;
constexpr int GT = 16;          // units per warp
constexpr int PT = 6;           // rows per lane
constexpr int ROWS = 32 * PT;   // rows per row-block
constexpr int NS = 3;           // time slices
constexpr int CH = 64;          // rows per staging chunk of the dW step

constexpr int cmax(int x, int y) { return x > y ? x : y; }

template <int H>
struct Geo {
    static constexpr int G = H / GT;               // warps per row-block
    static constexpr int RB = 8 / G;               // row-blocks per tile
    static constexpr int NROW = RB * ROWS;         // rows per tile
    static constexpr int PTS_RB = ROWS / NS;       // points per row-block
    static constexpr int PTS_TILE = RB * PTS_RB;   // points per tile
    static constexpr int ACT = RB * H * ROWS;      // floats of one layer's activations (24576 for every H)
    static constexpr int SCR = cmax(cmax(H * H, CH * (H + 1)), 4 * NROW);   // >= one weight layer, as k_mlp_deep's 2nd buffer
    static constexpr size_t SMEM = (size_t(ACT) + 5 * H + H * H + SCR) * sizeof(float);
};

__host__ __device__ constexpr size_t grad_len(int H, int L) {
    return size_t(9) * H + 4 + size_t(L - 1) * (size_t(H) * H + H);
}

template <int H>
__global__ void __launch_bounds__(NT, 1) k_deep_grad(const __grid_constant__ DeepGradArgs a) {
    using Q = Geo<H>;
    constexpr int G = Q::G, RB = Q::RB, NROW = Q::NROW, PTS_RB = Q::PTS_RB, PTS_TILE = Q::PTS_TILE, ACT = Q::ACT;
    constexpr int PPL = PT / NS;
    extern __shared__ __align__(16) float smem[];
    float* s_act = smem;                                              // [RB][H][ROWS]
    float2* s_l1 = reinterpret_cast<float2*>(smem + ACT);             // [5][H/2] layer-1 pairs (as k_mlp_deep)
    float* s_w = smem + ACT + 5 * H;                                  // [H][H] one hidden layer, k_mlp_deep's layout
    float* s_scr = s_w + H * H;                                       // staging: [CH][H+1] | y_bar / coords [NROW] float4
    float4* s_row = reinterpret_cast<float4*>(s_scr);
    __shared__ double s_red[NT / 32][6];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rb = warp / G, g0 = (warp % G) * GT;
    const int L = a.hidden_layers, nl = L - 1;
    const long long n_slab = (long long)(a.z_end - a.z_begin) * a.ny * a.nx;
    const long long tiles = (n_slab + PTS_TILE - 1) / PTS_TILE;
    const int plane = a.nx * a.ny;
    const long long qoff = (long long)(a.z_begin - a.z_origin) * plane;   // processed point -> residual index

    const size_t P = grad_len(H, L);
    const size_t oW1 = 0, ob1 = 4 * H, oWh = 5 * H, obh = oWh + size_t(nl) * H * H, oW2 = obh + size_t(nl) * H, ob2 = oW2 + 4 * H;
    double* part = a.partials + size_t(blockIdx.x) * (P + 2);
    float* ck = a.ckpt + size_t(blockIdx.x) * L * ACT;
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
        if (wcur != 0) load_layer(0);   // s_w is free: the previous tile's last contraction is behind a barrier
        // ================= forward ================================================================================
        // ---- layer 1 (k_mlp_deep's arithmetic) -> s_act and checkpoint 0 ----------------------------------------
        {
            float cx[PPL], cy[PPL], cz[PPL];
#pragma unroll
            for (int jp = 0; jp < PPL; ++jp) {
                long long p = tile * PTS_TILE + rb * PTS_RB + lane * PPL + jp;
                if (p > n_slab - 1) p = n_slab - 1;   // tail tile: a valid point, its y_bar is zero
                const int zl = int(p / plane), rem = int(p - (long long)zl * plane);
                const int y = rem / a.nx, x = rem - y * a.nx;
                cx[jp] = __ldg(a.cxs + x); cy[jp] = __ldg(a.cys + y); cz[jp] = __ldg(a.czs + a.z_begin + zl);
            }
            const int off = (rb * H) * ROWS + lane * PT;
            float* dst = s_act + off;
            float* dck = ck + off;
#pragma unroll 2
            for (int q = 0; q < GT / 2; ++q) {
                const int qq = g0 / 2 + q;
                const float2 b1p = s_l1[qq], w0s = s_l1[H / 2 + qq], w1s = s_l1[2 * (H / 2) + qq], w2s = s_l1[3 * (H / 2) + qq];
                const float2 w3 = s_l1[4 * (H / 2) + qq];
                const float2 tm = make_float2(__fmul_rn(w3.x, a.tc[0]), __fmul_rn(w3.y, a.tc[0]));
                const float2 t0 = make_float2(__fmul_rn(w3.x, a.tc[1]), __fmul_rn(w3.y, a.tc[1]));
                const float2 tp = make_float2(__fmul_rn(w3.x, a.tc[2]), __fmul_rn(w3.y, a.tc[2]));
#pragma unroll
                for (int jp = 0; jp < PPL; ++jp) {
                    const f32x2 sx = add2_rn_swapped(pack2(b1p), mul2_rn(pack2(w0s), bcast2(cx[jp])));
                    const f32x2 sxy = add2_rn_swapped(sx, mul2_rn(pack2(w1s), bcast2(cy[jp])));
                    const f32x2 sxyz = add2_rn_swapped(sxy, mul2_rn(pack2(w2s), bcast2(cz[jp])));
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        const float2 pt = s == 0 ? tm : (s == 1 ? t0 : tp);
                        float v0, v1;
                        unpack2(add2_rn(sxyz, pack2(pt)), v0, v1);
                        v0 = relu_ref(v0); v1 = relu_ref(v1);
                        dst[(2 * qq) * ROWS + jp * NS + s] = v0;
                        dst[(2 * qq + 1) * ROWS + jp * NS + s] = v1;
                        dck[(2 * qq) * ROWS + jp * NS + s] = v0;
                        dck[(2 * qq + 1) * ROWS + jp * NS + s] = v1;
                    }
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

        // ================= backward ===============================================================================
        // ---- y_bar of every row: A_t (slice t), +A_+ (t+dt), -A_+ (t-dt); zero for the tail rows --------------------
        for (int r = threadIdx.x; r < NROW; r += NT) {
            const int rbk = r / ROWS, row = r - rbk * ROWS, s = row % NS;
            const long long p = tile * PTS_TILE + rbk * PTS_RB + row / NS;
            float4 yb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p < n_slab) {
                const size_t qi = size_t(p + qoff);
                const float rq[4] = {__ldg(a.R[0] + qi), __ldg(a.R[1] + qi), __ldg(a.R[2] + qi), __ldg(a.R[3] + qi)};
                if (s == 1) {
                    yb = __ldg(a.adj + p);
                    red[4] += double(rq[0]) * double(rq[0]);
                    red[5] += double(rq[1]) * double(rq[1]) + double(rq[2]) * double(rq[2]) + double(rq[3]) * double(rq[3]);
                } else {
                    const float sg = s == 2 ? 1.f : -1.f;
                    yb = make_float4(sg * (a.scale_s * rq[0] * a.inv2dt), sg * (a.scale_u * rq[1] * a.inv2dt),
                                     sg * (a.scale_u * rq[2] * a.inv2dt), sg * (a.scale_u * rq[3] * a.inv2dt));
                }
                red[0] += double(yb.x); red[1] += double(yb.y); red[2] += double(yb.z); red[3] += double(yb.w);
            }
            s_row[r] = yb;
        }
        __syncthreads();
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
        // ---- layer 1: delta_z_1 = delta_a_1 (.) (a_1 > 0); dW1[h,:] += sum delta_z_1 (x, y, z, t_s), db1 += sum delta_z_1
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
                const int rbk = r / ROWS, row = r - rbk * ROWS;
                long long p = tile * PTS_TILE + rbk * PTS_RB + row / NS;
                if (p > n_slab - 1) p = n_slab - 1;
                const int zl = int(p / plane), rem = int(p - (long long)zl * plane);
                const int y = rem / a.nx, x = rem - y * a.nx;
                s_row[r] = make_float4(__ldg(a.cxs + x), __ldg(a.cys + y), __ldg(a.czs + a.z_begin + zl), a.tc[row % NS]);
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
    // db2 and the two residual sums: warps in order, then the block's slots
#pragma unroll
    for (int o = 0; o < 6; ++o) {
        const double v = warp_sum_d(red[o]);
        if (lane == 0) s_red[warp][o] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        double s = 0.0;
        for (int w = 0; w < NT / 32; ++w) s += s_red[w][threadIdx.x];
        part[threadIdx.x < 4 ? ob2 + threadIdx.x : P + (threadIdx.x - 4)] = s;
    }
}

// one thread per entry: block partials summed in block order
__global__ void k_deep_grad_reduce(const double* __restrict__ partials, int blocks, size_t P, double* grad, double* acc_out) {
    const size_t e = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= P + 2) return;
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += partials[size_t(b) * (P + 2) + e];
    if (e < P) grad[e] = s;
    else if (acc_out) acc_out[e - P] = s;
}

template <int H>
int launch_t(const DeepGradArgs& a, int blocks, double* grad, double* acc_out, cudaStream_t st) {
    constexpr size_t smem = Geo<H>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_deep_grad<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_deep_grad<H><<<blocks, NT, smem, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    const size_t P = grad_len(H, a.hidden_layers);
    k_deep_grad_reduce<<<unsigned((P + 2 + 255) / 256), 256, 0, st>>>(a.partials, blocks, P, grad, acc_out);
    return int(cudaGetLastError());
}

}  // namespace

size_t deep_grad_len(int H, int hidden_layers) {
    if ((H != 32 && H != 64 && H != 128) || hidden_layers < 1 || hidden_layers > 16) return 0;
    return grad_len(H, hidden_layers);
}

size_t deep_grad_ckpt_floats(int H, int hidden_layers) {
    (void)H;   // RB x H x ROWS = 8 x 16 x 192 for every width
    return size_t(hidden_layers) * Geo<32>::ACT;
}

int deep_grad_blocks(int H, long long n_points, int max_blocks) {
    const int pts = H == 32 ? Geo<32>::PTS_TILE : (H == 64 ? Geo<64>::PTS_TILE : Geo<128>::PTS_TILE);
    const long long tiles = (n_points + pts - 1) / pts;
    return int(tiles < max_blocks ? (tiles > 0 ? tiles : 1) : max_blocks);
}

int deep_grad_launch(int H, const DeepGradArgs& a, int blocks, double* grad, double* acc_out, cudaStream_t st) {
    switch (H) {
        case 32: return launch_t<32>(a, blocks, grad, acc_out, st);
        case 64: return launch_t<64>(a, blocks, grad, acc_out, st);
        case 128: return launch_t<128>(a, blocks, grad, acc_out, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
