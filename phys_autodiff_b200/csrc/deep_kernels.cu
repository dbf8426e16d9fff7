// Deeper coordinate MLPs over the grid, strict fp32, as a register-blocked contraction on the CUDA cores.
// See deep_kernels.cuh for what is computed and why parity for L > 1 is "unpinned".
//
// Governing roofline: the FP32 pipe in its non-contracted mode (every multiply and every add rounded
// separately, DESIGN.md section 4.1: 36.9 TFLOP/s measured).  A hidden->hidden layer costs 2*H*H lane-operations
// per point and slice, so everything else has to stay out of the FMA pipe's way:
//   * "rows" = (point, time slice) pairs: the three slices of a point go through the hidden layers as three
//     independent rows, so one weight fetch serves them all;
//   * a block of 8 warps holds, in shared memory, ONE layer's activations of its rows  act[row-block][h][192 rows]
//     (96 KB for every H) and the H x H weights of the current layer (and of the next one: cp.async
//     double buffer; for L <= 3 all hidden->hidden layers simply stay resident);
//   * a warp owns 16 consecutive outputs g of one row-block, a lane 6 rows: 96 accumulators as 48 packed
//     f32x2 pairs {g, g+1}.  Per input h it reads its 6 activations (3 x LDS.64, conflict-free) and the 16
//     weights W[g..g+15, h] (4 x LDS.128, one address per warp: broadcast) and issues 48 FMUL2 + 48 FADD2 --
//     7 shared-memory instructions per 96 packed math instructions (192 pipe cycles), where the previous kernel
//     (one point per thread, a uniform LDG.128 per two packed instructions) kept the LSU as busy as the pipe;
//   * the sum for output g starts at the bias and adds W[g,h]*a[h] for h ascending with FMUL2/FADD2 kept
//     un-contracted by the half-swap trick (mlp_eval.cuh): bit-identical to the CPU restatement;
//   * outputs replace the inputs IN PLACE (the accumulators hold the whole layer's outputs of the warp, so one
//     block barrier separates "everybody has read layer l" from "write layer l+1"): one activation buffer, which
//     is what lets H = 128 fit (96 KB + 2 x 64 KB) without ever keeping 128 activations in registers.
//   H = 128: 8 output groups x 1 row-block of 192 rows;  H = 64: 4 x 2;  H = 32: 2 x 4.
// Layer 1 (4 -> H) and the output layer (H -> 4) are 1/32 .. 1/8 of one hidden->hidden layer and run as
// plain strict-fp32 phases on the same shared-memory activations (weights from the kernel-parameter constant
// bank, MlpConst<H>, exactly as the one-hidden-layer kernels: L = 1 is bit-identical to them).
// Points mode (POINTS = true, deep_points_launch) is the same kernel with one time slice whose rows are caller-supplied
// inputs: one float4 load per row instead of the three coordinate-table loads, W1[h,3] * t rounded per row.
#include "deep_kernels.cuh"
#include "mlp_eval.cuh"

#include <cstdlib>

namespace physad {

namespace {

__device__ __forceinline__ unsigned smem_addr(const void* p) { return unsigned(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int DEEP_THREADS = 256;
constexpr int GT = 16;          // outputs per warp
constexpr int PT = 6;           // rows per lane
constexpr int ROWS = 32 * PT;   // rows per row-block

// POINTS: rows are the caller's points a.pts[0 .. n_points) (AoS {x, y, z, t}, one time slice), outputs to out_aos
template <int H, bool FIELDS, int VAR, bool POINTS>
__global__ void __launch_bounds__(DEEP_THREADS, 1) k_mlp_deep(const __grid_constant__ MlpConst<H> w, const __grid_constant__ DeepArgs a) {
    static_assert(!(POINTS && FIELDS), "points mode writes AoS outputs");
    constexpr int G = H / GT;              // output groups = warps per row-block
    constexpr int RB = 8 / G;              // row-blocks per block
    constexpr int NS = FIELDS ? 3 : 1;     // time slices
    constexpr int PPL = PT / NS;           // points per lane
    constexpr int PTS_RB = 32 * PPL;       // points per row-block
    constexpr int PTS_TILE = RB * PTS_RB;  // points per block tile
    static_assert(G * RB == 8 && PT % NS == 0, "8 warps; a lane's rows are whole points");
    extern __shared__ __align__(16) float smem[];
    float* s_act = smem;                   // [RB][H][ROWS]
    float2* s_l1 = reinterpret_cast<float2*>(smem + RB * H * ROWS);   // [5][H/2] layer-1 pairs, see below
    float* s_w = smem + RB * H * ROWS + 5 * H;   // [1 or 2][H][H], input-major: s_w[h*H + g], pairs stored (g+1, g)

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rb = warp / G, g0 = (warp % G) * GT;
    const int nl = a.hidden_layers - 1;    // hidden->hidden layers
    const bool resident = nl <= 2;         // both buffers hold a layer for good
    const long long n_slab = POINTS ? a.n_points : (long long)(a.z_end - a.z_begin) * a.ny * a.nx;
    const long long tiles = (n_slab + PTS_TILE - 1) / PTS_TILE;
    const int plane = a.nx * a.ny;

    auto load_layer = [&](int buf, int layer) {
        const float* src = a.wh + size_t(layer) * H * H;
        float* dst = s_w + buf * H * H;
        for (int i = threadIdx.x; i < H * H / 4; i += DEEP_THREADS) cp_async16(dst + 4 * i, src + 4 * i);
    };
    // streaming: step c (over this block's tiles x layers) uses buffer c & 1 and layer c % nl
    long long my_tiles = blockIdx.x < tiles ? (tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const long long steps = my_tiles * nl;
    long long c = 0;
    // layer-1 weights per PAIR of hidden units (2q, 2q+1), staged once: a warp indexes them by ITS units, which the
    // compiler cannot prove warp-uniform -- from the constant bank that is a per-thread LDC (slow path), from shared
    // memory a broadcast LDS.  [0] {b1} | [1..3] {W1[.,0..2]} half-swapped (mlp_eval.cuh) | [4] {W1[.,3]}
    for (int q = threadIdx.x; q < H / 2; q += DEEP_THREADS) {
        const float4 ra = __ldg(reinterpret_cast<const float4*>(a.W1) + 2 * q), rb4 = __ldg(reinterpret_cast<const float4*>(a.W1) + 2 * q + 1);
        s_l1[q] = make_float2(__ldg(a.b1 + 2 * q), __ldg(a.b1 + 2 * q + 1));
        s_l1[H / 2 + q] = make_float2(rb4.x, ra.x);
        s_l1[2 * (H / 2) + q] = make_float2(rb4.y, ra.y);
        s_l1[3 * (H / 2) + q] = make_float2(rb4.z, ra.z);
        s_l1[4 * (H / 2) + q] = make_float2(ra.w, rb4.w);
    }
    __syncthreads();
    if (nl > 0 && my_tiles > 0) {
        load_layer(0, 0);
        cp_async_commit();
        if (nl > 1 || !resident) {
            if (steps > 1) load_layer(1, 1 % nl);
            cp_async_commit();
        }
    }

    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        // ---- layer 1: this warp's 16 hidden units for its lane's points, all slices -> s_act ------------------
        {
            float cx[PPL], cy[PPL], cz[PPL], ct[PPL];
#pragma unroll
            for (int jp = 0; jp < PPL; ++jp) {
                long long p = tile * PTS_TILE + rb * PTS_RB + lane * PPL + jp;
                if (p > n_slab - 1) p = n_slab - 1;   // tail tile: evaluate a valid point, never stored
                if (POINTS) {
                    const float4 c4 = __ldg(a.pts + p);
                    cx[jp] = c4.x; cy[jp] = c4.y; cz[jp] = c4.z; ct[jp] = c4.w;
                } else {
                    const int zl = int(p / plane), rem = int(p - (long long)zl * plane);
                    const int y = rem / a.nx, x = rem - y * a.nx;
                    cx[jp] = __ldg(a.cxs + x); cy[jp] = __ldg(a.cys + y); cz[jp] = __ldg(a.czs + a.z_begin + zl);
                }
            }
            float* dst = s_act + (rb * H) * ROWS + lane * PT;
#pragma unroll 2
            for (int q = 0; q < GT / 2; ++q) {
                const int qq = g0 / 2 + q;
                const float2 b1p = s_l1[qq], w0s = s_l1[H / 2 + qq], w1s = s_l1[2 * (H / 2) + qq], w2s = s_l1[3 * (H / 2) + qq];
                const float2 w3 = s_l1[4 * (H / 2) + qq];
                // W1[h,3] * t_slice, rounded separately -- the same IEEE product the host pre-rounds for MlpConst::pt*
                const float2 tm = make_float2(__fmul_rn(w3.x, a.tc[0]), __fmul_rn(w3.y, a.tc[0]));
                const float2 t0 = make_float2(__fmul_rn(w3.x, a.tc[1]), __fmul_rn(w3.y, a.tc[1]));
                const float2 tp = make_float2(__fmul_rn(w3.x, a.tc[2]), __fmul_rn(w3.y, a.tc[2]));
#pragma unroll
                for (int jp = 0; jp < PPL; ++jp) {
                    // ((b1 + W1[.,0] x) + W1[.,1] y) + W1[.,2] z, then + the pre-rounded W1[.,3] t_slice (mlp_eval.cuh)
                    const f32x2 sx = add2_rn_swapped(pack2(b1p), mul2_rn(pack2(w0s), bcast2(cx[jp])));
                    const f32x2 sxy = add2_rn_swapped(sx, mul2_rn(pack2(w1s), bcast2(cy[jp])));
                    const f32x2 sxyz = add2_rn_swapped(sxy, mul2_rn(pack2(w2s), bcast2(cz[jp])));
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        // points mode: the row's own t, the product rounded per row
                        const float2 pt = POINTS ? make_float2(__fmul_rn(w3.x, ct[jp]), __fmul_rn(w3.y, ct[jp]))
                                                 : (NS == 1 ? t0 : (s == 0 ? tm : (s == 1 ? t0 : tp)));
                        float v0, v1;
                        unpack2(add2_rn(sxyz, pack2(pt)), v0, v1);
                        dst[(2 * qq) * ROWS + jp * NS + s] = relu_ref(v0);
                        dst[(2 * qq + 1) * ROWS + jp * NS + s] = relu_ref(v1);
                    }
                }
            }
        }
        if (nl > 0 && resident && tile == blockIdx.x) cp_async_wait<0>();   // resident weights: landed once
        __syncthreads();

        // ---- hidden -> hidden layers ---------------------------------------------------------------------------
        for (int l = 0; l < nl; ++l, ++c) {
            if (!resident) {
                cp_async_wait<1>();   // step c's weights have landed (only step c+1's group may still be in flight)
                __syncthreads();
            }
            const float* wbuf = s_w + (resident ? l : int(c & 1)) * H * H + g0;
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
            auto load_h = [&](int h, float (&av)[PT], float4 (&wv)[GT / 4]) {
#pragma unroll
                for (int j = 0; j < PT; j += 2) {
                    const float2 t = *reinterpret_cast<const float2*>(arow + h * ROWS + j);
                    av[j] = t.x; av[j + 1] = t.y;
                }
#pragma unroll
                for (int v = 0; v < GT / 4; ++v) wv[v] = *reinterpret_cast<const float4*>(wbuf + h * H + 4 * v);
            };
            auto math_h = [&](const float (&av)[PT], const float4 (&wv)[GT / 4]) {
#pragma unroll
                for (int j = 0; j < PT; ++j) {
                    const f32x2 aa = bcast2(av[j]);
#pragma unroll
                    for (int v = 0; v < GT / 4; ++v) {   // {W[g+1,h], W[g,h], W[g+3,h], W[g+2,h]}
                        q[j][2 * v] = add2_rn_swapped(q[j][2 * v], mul2_rn(aa, pack2(wv[v].x, wv[v].y)));
                        q[j][2 * v + 1] = add2_rn_swapped(q[j][2 * v + 1], mul2_rn(aa, pack2(wv[v].z, wv[v].w)));
                    }
                }
            };
            if (VAR == 0) {
#pragma unroll 2
                for (int h = 0; h < H; ++h) {
                    float av[PT];
                    float4 wv[GT / 4];
                    load_h(h, av, wv);
                    math_h(av, wv);
                }
            } else {
#pragma unroll 4
                for (int h = 0; h < H; ++h) {
                    float av[PT];
                    float4 wv[GT / 4];
                    load_h(h, av, wv);
                    math_h(av, wv);
                }
            }
            __syncthreads();   // every warp has read this layer's inputs (and this weight buffer)
            if (!resident && c + 2 < steps) load_layer(int(c & 1), int((c + 2) % nl));
            if (!resident) cp_async_commit();
            {
                float* orow = s_act + (rb * H + g0) * ROWS + lane * PT;
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
                        *reinterpret_cast<float2*>(orow + (2 * p) * ROWS + j) = make_float2(lo[j], lo[j + 1]);
                        *reinterpret_cast<float2*>(orow + (2 * p + 1) * ROWS + j) = make_float2(hi[j], hi[j + 1]);
                    }
                }
            }
            __syncthreads();
        }

        // ---- output layer: a thread takes one row at a time (RB*192 rows over 256 threads) and forms its four outputs
        // as two packed pairs, h ascending, weight pairs straight from the constant bank -- the arithmetic of
        // mlp_eval's layer 2, so L = 1 equals the one-hidden-layer kernels bit for bit -------------------------------
        {
            constexpr int NROW = RB * ROWS, PASSES = (NROW + DEEP_THREADS - 1) / DEEP_THREADS;
            const float4 b2 = w.b2;
            const size_t n = size_t(n_slab);
#pragma unroll
            for (int pass = 0; pass < PASSES; ++pass) {
                const int rowg_raw = threadIdx.x + DEEP_THREADS * pass;
                const int rowg = rowg_raw < NROW ? rowg_raw : NROW - 1;   // idle threads of the last pass redo a row: the loop
                {                                                          // stays convergent, so W2 arrives by uniform loads
                    const int rbk = rowg / ROWS, row = rowg - rbk * ROWS;
                    const float* src = s_act + (rbk * H) * ROWS + row;
                    f32x2 q01 = pack2(b2.x, b2.y), q23 = pack2(b2.z, b2.w);
#pragma unroll   // fully: compile-time constant-bank offsets (a rolled loop gets per-thread LDC here, the slow path)
                    for (int h = 0; h < H; ++h) {
                        const float4 cw = w.w2[h];   // {W2[1,h], W2[0,h], W2[3,h], W2[2,h]}
                        const f32x2 aa = bcast2(src[h * ROWS]);
                        q01 = add2_rn_swapped(q01, mul2_rn(aa, pack2(cw.x, cw.y)));
                        q23 = add2_rn_swapped(q23, mul2_rn(aa, pack2(cw.z, cw.w)));
                    }
                    float y0, y1, y2, y3;
                    unpack2(q01, y0, y1);
                    unpack2(q23, y2, y3);
                    const long long i = tile * PTS_TILE + rbk * PTS_RB + row / NS;
                    if (i < n_slab && rowg_raw < NROW) {
                        if (FIELDS) {
                            const int sl = row % NS;
                            a.sigma[sl][i] = y0;
                            a.u[sl][i] = y1;
                            a.u[sl][n + i] = y2;
                            a.u[sl][2 * n + i] = y3;
                        } else {
                            a.out_aos[i] = make_float4(y0, y1, y2, y3);
                        }
                    }
                }
            }
        }
        __syncthreads();   // the next tile's layer 1 overwrites s_act
    }
    cp_async_wait<0>();
}

template <int H>
size_t smem_for(int hidden_layers) {
    const int nl = hidden_layers - 1;
    const size_t act = size_t(8 / (H / GT)) * H * ROWS * sizeof(float) + size_t(5) * H * sizeof(float);   // + layer-1 pairs
    const size_t wbuf = size_t(nl == 0 ? 0 : (nl == 1 ? 1 : 2)) * H * H * sizeof(float);
    return act + wbuf;
}

template <int H, bool FIELDS, int VAR, bool POINTS = false>
int launch_v(const void* mlp_const, const DeepArgs& a, int grid_blocks, cudaStream_t st) {
    const size_t smem = smem_for<H>(a.hidden_layers);
    cudaError_t e = cudaFuncSetAttribute(k_mlp_deep<H, FIELDS, VAR, POINTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_mlp_deep<H, FIELDS, VAR, POINTS><<<grid_blocks, DEEP_THREADS, smem, st>>>(*static_cast<const MlpConst<H>*>(mlp_const), a);
    return int(cudaGetLastError());
}

template <int H, bool FIELDS>
int launch_t(const void* mlp_const, const DeepArgs& a, int grid_blocks, cudaStream_t st) {
    // measured at 256^3 (profiles/r02_deep_variants.json): unroll 4 beats unroll 2 by 1-5 %; an explicit two-stage
    // software pipeline of the operand loads was 10-15 % slower (240 registers, worse schedule) and is not built
    static const int var = getenv("PHYSAD_DEEP_VARIANT") ? atoi(getenv("PHYSAD_DEEP_VARIANT")) : 1;   // tuning aid
    return var == 0 ? launch_v<H, FIELDS, 0>(mlp_const, a, grid_blocks, st) : launch_v<H, FIELDS, 1>(mlp_const, a, grid_blocks, st);
}

}  // namespace

size_t deep_smem_bytes(int H, int hidden_layers) {
    return H == 32 ? smem_for<32>(hidden_layers) : (H == 64 ? smem_for<64>(hidden_layers) : smem_for<128>(hidden_layers));
}

int deep_launch(int H, bool fields, const void* mlp_const, const DeepArgs& a, int grid_blocks, cudaStream_t st) {
    switch (H) {
        case 32: return fields ? launch_t<32, true>(mlp_const, a, grid_blocks, st) : launch_t<32, false>(mlp_const, a, grid_blocks, st);
        case 64: return fields ? launch_t<64, true>(mlp_const, a, grid_blocks, st) : launch_t<64, false>(mlp_const, a, grid_blocks, st);
        case 128: return fields ? launch_t<128, true>(mlp_const, a, grid_blocks, st) : launch_t<128, false>(mlp_const, a, grid_blocks, st);
    }
    return int(cudaErrorInvalidValue);
}

int deep_points_launch(int H, const void* mlp_const, const DeepArgs& a, int grid_blocks, cudaStream_t st) {
    switch (H) {   // the unroll-4 variant only (launch_t's default)
        case 32: return launch_v<32, false, 1, true>(mlp_const, a, grid_blocks, st);
        case 64: return launch_v<64, false, 1, true>(mlp_const, a, grid_blocks, st);
        case 128: return launch_v<128, false, 1, true>(mlp_const, a, grid_blocks, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
