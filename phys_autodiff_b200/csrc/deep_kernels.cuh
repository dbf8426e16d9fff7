// Deeper coordinate MLPs (BASELINE config 5: width / depth sweep): In = 4 -> H -> H -> ... -> H -> Out = 4 with
// L >= 1 hidden layers, H in {32, 64, 128}.  ADDITIVE: the reference API (include/mlp.h:5-6) has exactly one
// hidden layer, so for L > 1 there is no reference implementation to pin against -- the semantics are the
// reference's layer rule applied again (src/mlp_cpu.cpp:19-24: start from the bias, add W[g,h]*a[h] for h
// ascending, separate fp32 multiply and add, ReLU), restated for the CPU by the test oracle
// (oracle_mlp_forward_deep, "parity unpinned" for L > 1; L = 1 is pinned: it must equal the one-hidden-layer
// path bit for bit, and the tests check that).  The reference names the target in REQUIREMENT.md:157
// (tiny-cuda-nn-style fused MLP) and docs/PLAN_MLP_SMOKE_INTEGRATION.md:49-51.
//
// Interface of deep_kernels.cu (its own translation unit).
#pragma once
#include <cuda_runtime.h>

namespace physad {

struct DeepArgs {
    int nx, ny, nz;
    int z_begin, z_end;
    int hidden_layers;          // L >= 1
    const float* cxs; const float* cys; const float* czs;
    const float* W1;            // [H][4] device copy in the reference's layout (layer 1 is staged in shared memory from it)
    const float* b1;            // [H]
    float tc[3];                // network time input of the slices t-dt, t, t+dt (grid infer: tc[1])
    const float* wh;            // [(L-1)][H][H]: for layer l and INPUT h, the H outputs with pairs stored (g+1, g)
    const float* bh;            // [(L-1)][H]
    float4* out_aos;            // FIELDS = false: [slab points] {sigma, ux, uy, uz}
    float* sigma[3];            // FIELDS = true: t-dt, t, t+dt
    float* u[3];                //   channel-major, channel stride = slab points
    // points mode (deep_points_launch): the rows are n_points caller-supplied inputs {x, y, z, t}, outputs to out_aos
    const float4* pts;
    long long n_points;
};

// `mlp_const` points to a host MlpConst<H> (mlp_eval.cuh) for the template width H in {32, 64, 128}.
// Returns a cudaError_t value.  grid_blocks: persistent grid size (normally the SM count).
int deep_launch(int H, bool fields, const void* mlp_const, const DeepArgs& a, int grid_blocks, cudaStream_t st);
// The same kernel with its rows taken from a.pts (one float4 load per row) instead of the grid index: the network at
// a.n_points arbitrary points, out_aos[i] = MLP(pts[i]).  Layer 1 forms W1[h,3] * t per row (the grid modes use the
// same IEEE product per slice), so at grid coordinates the outputs equal the grid mode's bit for bit.  a.nx .. a.tc,
// a.sigma and a.u are not read.
int deep_points_launch(int H, const void* mlp_const, const DeepArgs& a, int grid_blocks, cudaStream_t st);
// Dynamic shared memory the kernel needs for (H, hidden_layers), for diagnostics / tests.
size_t deep_smem_bytes(int H, int hidden_layers);

}  // namespace physad
