// See tangent_grad_kernels.cuh.
#include "tangent_grad_kernels.cuh"

#include "mlp_eval.cuh"
#include "tangent_kernels.cuh"

namespace physad {

namespace {

__device__ __forceinline__ double warp_sum_dbl(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int HT>
__global__ void __launch_bounds__(TGRAD_THREADS, 2) k_tangent_grad(const __grid_constant__ TangentConst<HT> w, const TangentGradArgs a) {
    static_assert(TGRAD_THREADS % HT == 0 && HT % 32 == 0, "a warp's lanes are 32 hidden units of one point group");
    constexpr int NGRP = TGRAD_THREADS / HT;           // point groups of a chunk, HT points each
    constexpr int NGT = TGRAD_NACC * HT + 6;           // partial: [24][HT] per-unit sums, db2[4], the two square sums
    static_assert(TGRAD_NACC * HT <= 6 * TGRAD_THREADS * 2, "the last block's totals fit the staging arrays");
    // staged per point: {cx, cy, cz, 0} | yb[4] | Jb[o][0..3] for o = 0..3   (24 KB, reused by the reductions)
    __shared__ float4 s_st[6][TGRAD_THREADS];
    __shared__ double s_misc[TGRAD_THREADS / 32 * 6];
    __shared__ unsigned int s_flag;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int hu = tid % HT, grp = tid / HT;
    const long long n = (long long)(a.z_end - a.z_begin) * a.ny * a.nx;
    const long long nch = (n + TGRAD_THREADS - 1) / TGRAD_THREADS;
    const int plane = a.nx * a.ny;
    // this thread's hidden unit, as the forward forms z_h (padded units are zero records: z = 0, mask 0)
    const float4 w1 = w.w1[hu], w2 = w.w2[hu];
    const float b1 = w.b1[hu];

    double D[TGRAD_NACC];
#pragma unroll
    for (int k = 0; k < TGRAD_NACC; ++k) D[k] = 0.0;
    double db2[4] = {0.0, 0.0, 0.0, 0.0}, acc_s = 0.0, acc_u = 0.0;

    for (long long ch = blockIdx.x; ch < nch; ch += gridDim.x) {
        // ---- stage: thread per point ------------------------------------------------------------------------------
        {
            const long long p = ch * TGRAD_THREADS + tid;
            float4 st[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) st[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p < n) {
                const int zl = int(p / plane), rem = int(p - (long long)zl * plane);
                const int yy = rem / a.nx, xx = rem - yy * a.nx;
                const float cx = __ldg(a.cxs + xx), cy = __ldg(a.cys + yy), cz = __ldg(a.czs + a.z_begin + zl);
                float y[4] = {w.b2.x, w.b2.y, w.b2.z, w.b2.w};
                f32x2 Ja[4] = {0ull, 0ull, 0ull, 0ull}, Jb[4] = {0ull, 0ull, 0ull, 0ull};   // {J[o][0], J[o][1]}, {J[o][2], J[o][3]}
#pragma unroll 4
                for (int h = 0; h < HT; ++h) {
                    const float4 v1 = w.w1[h], v2 = w.w2[h];
                    // k_tangent_loss's roundings in its order: ((b1 + W1x cx) + W1y cy) + W1z cz, then + fl(W1t ct)
                    float z = __fadd_rn(w.b1[h], __fmul_rn(v1.x, cx));
                    z = __fadd_rn(z, __fmul_rn(v1.y, cy));
                    z = __fadd_rn(z, __fmul_rn(v1.z, cz));
                    z = __fadd_rn(z, v1.w);
                    const float act = fmaxf(z, 0.f);
                    y[0] = __fmaf_rn(v2.x, act, y[0]);
                    y[1] = __fmaf_rn(v2.y, act, y[1]);
                    y[2] = __fmaf_rn(v2.z, act, y[2]);
                    y[3] = __fmaf_rn(v2.w, act, y[3]);
                    // fma(m, p, J) with m in {0, 1} is J + p or J: the same bits as the forward's packed fma
                    if (z > 0.f) {
#pragma unroll
                        for (int o = 0; o < 4; ++o) {
                            const float4 pv = w.p[h][o];
                            Ja[o] = add2_rn(Ja[o], pack2(pv.x, pv.y));
                            Jb[o] = add2_rn(Jb[o], pack2(pv.z, pv.w));
                        }
                    }
                }
                float J[4][4];
#pragma unroll
                for (int o = 0; o < 4; ++o) {
                    unpack2(Ja[o], J[o][0], J[o][1]);
                    unpack2(Jb[o], J[o][2], J[o][3]);
                }
                // residuals: the expressions of k_tangent_loss
                const float s[3] = {a.sx, a.sy, a.sz};
                float g[4][3];
#pragma unroll
                for (int o = 0; o < 4; ++o)
#pragma unroll
                    for (int j = 0; j < 3; ++j) g[o][j] = J[o][j] * s[j];
                const float div = (g[1][0] + g[2][1]) + g[3][2];
                float R[4];
#pragma unroll
                for (int o = 0; o < 4; ++o) R[o] = J[o][3] + ((y[1] * g[o][0] + y[2] * g[o][1]) + y[3] * g[o][2]);
                R[0] += y[0] * div;
                acc_s += double(R[0]) * double(R[0]);
                acc_u += double(R[1]) * double(R[1]) + double(R[2]) * double(R[2]) + double(R[3]) * double(R[3]);
                // adjoints
                float gb[4];
                gb[0] = a.scale_s * R[0];
#pragma unroll
                for (int o = 1; o < 4; ++o) gb[o] = a.scale_u * R[o];
                float yb[4];
                yb[0] = gb[0] * div;
#pragma unroll
                for (int j = 0; j < 3; ++j) yb[j + 1] = ((gb[0] * g[0][j] + gb[1] * g[1][j]) + gb[2] * g[2][j]) + gb[3] * g[3][j];
                const float gy0 = gb[0] * y[0];
                float jb[4][4];
#pragma unroll
                for (int o = 0; o < 4; ++o) {
#pragma unroll
                    for (int j = 0; j < 3; ++j) jb[o][j] = s[j] * (o == j + 1 ? gb[o] * y[j + 1] + gy0 : gb[o] * y[j + 1]);
                    jb[o][3] = gb[o];
                }
                st[0] = make_float4(cx, cy, cz, 0.f);
                st[1] = make_float4(yb[0], yb[1], yb[2], yb[3]);
#pragma unroll
                for (int o = 0; o < 4; ++o) st[2 + o] = make_float4(jb[o][0], jb[o][1], jb[o][2], jb[o][3]);
#pragma unroll
                for (int o = 0; o < 4; ++o) db2[o] += double(yb[o]);
            }
            __syncthreads();   // the previous chunk's backward has read the staging arrays
#pragma unroll
            for (int k = 0; k < 6; ++k) s_st[k][tid] = st[k];
            __syncthreads();
        }
        // ---- backward: thread per (hidden unit hu, points grp*HT ... grp*HT + HT - 1) ----------------------------
#pragma unroll 1
        for (int i0 = grp * HT; i0 < grp * HT + HT; i0 += 32) {
            f32x2 S[4][2];                     // {S[o][0], S[o][1]}, {S[o][2], S[o][3]}
            float F[8];                        // sum yb_o a (4) | sum dz c_x, c_y, c_z | sum dz
#pragma unroll
            for (int o = 0; o < 4; ++o) S[o][0] = S[o][1] = 0ull;
#pragma unroll
            for (int k = 0; k < 8; ++k) F[k] = 0.f;
#pragma unroll 4
            for (int i = i0; i < i0 + 32; ++i) {
                const float4 c = s_st[0][i], yb = s_st[1][i];   // every lane reads the same point: broadcast
                // the forward's operation order: the same mask as the stage phase and the loss
                float z = __fadd_rn(b1, __fmul_rn(w1.x, c.x));
                z = __fadd_rn(z, __fmul_rn(w1.y, c.y));
                z = __fadd_rn(z, __fmul_rn(w1.z, c.z));
                z = __fadd_rn(z, w1.w);
                const bool m = z > 0.f;
                const float act = m ? z : 0.f;
                const float da = __fmaf_rn(w2.w, yb.w, __fmaf_rn(w2.z, yb.z, __fmaf_rn(w2.y, yb.y, w2.x * yb.x)));
                const float dz = m ? da : 0.f;
                F[0] = __fmaf_rn(yb.x, act, F[0]);
                F[1] = __fmaf_rn(yb.y, act, F[1]);
                F[2] = __fmaf_rn(yb.z, act, F[2]);
                F[3] = __fmaf_rn(yb.w, act, F[3]);
                F[4] = __fmaf_rn(dz, c.x, F[4]);
                F[5] = __fmaf_rn(dz, c.y, F[5]);
                F[6] = __fmaf_rn(dz, c.z, F[6]);
                F[7] += dz;
                if (m) {
#pragma unroll
                    for (int o = 0; o < 4; ++o) {
                        const float4 jb = s_st[2 + o][i];
                        S[o][0] = add2_rn(S[o][0], pack2(jb.x, jb.y));
                        S[o][1] = add2_rn(S[o][1], pack2(jb.z, jb.w));
                    }
                }
            }
#pragma unroll
            for (int o = 0; o < 4; ++o) {
                float lo, hi;
                unpack2(S[o][0], lo, hi);
                D[o * 4 + 0] += double(lo); D[o * 4 + 1] += double(hi);
                unpack2(S[o][1], lo, hi);
                D[o * 4 + 2] += double(lo); D[o * 4 + 3] += double(hi);
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) D[16 + k] += double(F[k]);
        }
    }

    // ---- block partial: the NGRP groups of each unit summed in group order, through shared memory ---------------
    double* part = a.partials + size_t(blockIdx.x) * NGT;
    double* s_red = reinterpret_cast<double*>(&s_st[0][0]);   // 3072 doubles
    constexpr int KP = 12;                                     // accumulators per pass: KP * 256 doubles = 24 KB
    __syncthreads();
#pragma unroll
    for (int k0 = 0; k0 < TGRAD_NACC; k0 += KP) {
#pragma unroll
        for (int k = 0; k < KP; ++k) s_red[k * TGRAD_THREADS + tid] = D[k0 + k];
        __syncthreads();
        for (int e = tid; e < KP * HT; e += TGRAD_THREADS) {
            const int k = e / HT, h = e - k * HT;
            double v = 0.0;
#pragma unroll
            for (int q = 0; q < NGRP; ++q) v += s_red[k * TGRAD_THREADS + q * HT + h];
            part[(k0 + k) * HT + h] = v;
        }
        __syncthreads();
    }
    const double misc[6] = {db2[0], db2[1], db2[2], db2[3], acc_s, acc_u};
#pragma unroll
    for (int o = 0; o < 6; ++o) {
        const double v = warp_sum_dbl(misc[o]);
        if (lane == 0) s_misc[wid * 6 + o] = v;
    }
    __syncthreads();
    if (tid < 6) {
        double v = 0.0;
#pragma unroll
        for (int q = 0; q < TGRAD_THREADS / 32; ++q) v += s_misc[q * 6 + tid];
        part[TGRAD_NACC * HT + tid] = v;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_flag = atomicAdd(a.ticket, 1u);
    __syncthreads();
    if (s_flag != gridDim.x - 1) return;
    __threadfence();

    // ---- last block: block-ordered totals, then the contraction into the reference layouts (runtime width) ----------
    double* tot = s_red;   // [24][HT]
    for (int e = tid; e < TGRAD_NACC * HT; e += TGRAD_THREADS) {
        double v = 0.0;
        for (unsigned int b = 0; b < gridDim.x; ++b) v += __ldcg(a.partials + size_t(b) * NGT + e);
        tot[e] = v;
    }
    if (tid < 6) {
        double v = 0.0;
        for (unsigned int b = 0; b < gridDim.x; ++b) v += __ldcg(a.partials + size_t(b) * NGT + TGRAD_NACC * HT + tid);
        s_misc[tid] = v;
    }
    __syncthreads();
    const int H = a.H;
    auto S = [&](int o, int k, int h) { return tot[(o * 4 + k) * HT + h]; };
    for (int e = tid; e < 9 * H + 4; e += TGRAD_THREADS) {
        double v;
        if (e < 4 * H) {                       // dW1[h,k]
            const int h = e >> 2, k = e & 3;
            v = k < 3 ? tot[(20 + k) * HT + h] : double(a.ct) * tot[23 * HT + h];
#pragma unroll
            for (int o = 0; o < 4; ++o) v += double(__ldg(a.W2 + o * H + h)) * S(o, k, h);
        } else if (e < 5 * H) {                // db1[h]
            v = tot[23 * HT + (e - 4 * H)];
        } else if (e < 9 * H) {                // dW2[o,h]
            const int o = (e - 5 * H) / H, h = (e - 5 * H) - o * H;
            v = tot[(16 + o) * HT + h];
#pragma unroll
            for (int k = 0; k < 4; ++k) v += double(__ldg(a.W1 + h * 4 + k)) * S(o, k, h);
        } else {                               // db2[o]
            v = s_misc[e - 9 * H];
        }
        a.grad[e] = v;
    }
    if (tid < 2) a.acc[tid] = s_misc[4 + tid];
    if (tid == 0) *a.ticket = 0u;
}

template <int HT>
int blocks_per_sm_t(int* out) {
    return int(cudaOccupancyMaxActiveBlocksPerMultiprocessor(out, k_tangent_grad<HT>, TGRAD_THREADS, 0));
}

template <int HT>
int launch_t(const void* k, const TangentGradArgs& a, unsigned blocks, cudaStream_t st) {
    k_tangent_grad<HT><<<blocks, TGRAD_THREADS, 0, st>>>(*static_cast<const TangentConst<HT>*>(k), a);
    return int(cudaGetLastError());
}

}  // namespace

int tangent_grad_blocks_per_sm(int HT, int* out) {
    switch (HT) {
        case 32: return blocks_per_sm_t<32>(out);
        case 64: return blocks_per_sm_t<64>(out);
        case 128: return blocks_per_sm_t<128>(out);
    }
    return int(cudaErrorInvalidValue);
}

int tangent_grad_launch(int HT, const void* tangent_const, const TangentGradArgs& a, unsigned blocks, cudaStream_t st) {
    switch (HT) {
        case 32: return launch_t<32>(tangent_const, a, blocks, st);
        case 64: return launch_t<64>(tangent_const, a, blocks, st);
        case 128: return launch_t<128>(tangent_const, a, blocks, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
