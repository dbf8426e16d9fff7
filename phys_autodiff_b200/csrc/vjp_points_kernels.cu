// The vector-Jacobian product of deep networks at points; see deep_data_kernels.cuh for what it computes and
// deep_data_body.cuh for the kernel, k_vjp_points<H>, whose source k_deep_data_grad shares.  A translation unit of its own,
// so the data kernels' object keeps exactly its three instantiations and the reduction, which this file reuses through
// deep_data_reduce.
#define DEEP_DATA_KERNEL k_vjp_points
#define DEEP_DATA_PAIRS false
#define DEEP_DATA_VJP true
#include "deep_data_body.cuh"

namespace physad {

namespace {

template <int H>
int launch_v(const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    constexpr size_t smem = Geo<H>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_vjp_points<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_vjp_points<H><<<blocks, NT, smem, st>>>(*static_cast<const MlpConst<H>*>(mlp_const), a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    return deep_data_reduce(a.partials, blocks, grad_len(H, a.hidden_layers), grad, acc, st);
}

}  // namespace

int vjp_points_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    switch (H) {
        case 32: return launch_v<32>(mlp_const, a, blocks, grad, acc, st);
        case 64: return launch_v<64>(mlp_const, a, blocks, grad, acc, st);
        case 128: return launch_v<128>(mlp_const, a, blocks, grad, acc, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
