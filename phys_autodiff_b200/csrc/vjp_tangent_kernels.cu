// The vector-Jacobian product of deep networks and their Jacobian at points; see deep_tangent_kernels.cuh for what it
// computes and deep_tangent_body.cuh for the kernel, k_vjp_tangent<H, true>, whose source k_colloc_tangent shares.  A
// translation unit of its own, so the other three objects keep exactly their instantiations.
#define DEEP_TANGENT_KERNEL k_vjp_tangent
#define DEEP_TANGENT_POINTS true
#define DEEP_TANGENT_VJP true
#include "deep_tangent_body.cuh"

namespace physad {

namespace {

template <int H>
int launch_v(const DeepTangentArgs& a, int blocks, double* acc, double* grad, cudaStream_t st) {
    constexpr size_t smem = Geo<H, true>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_vjp_tangent<H, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_vjp_tangent<H, true><<<blocks, NT, smem, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    return deep_tangent_reduce(a.partials, blocks, grad_len(H, a.hidden_layers), acc, grad, st);
}

}  // namespace

int vjp_tangent_launch(int H, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st) {
    switch (H) {
        case 32: return launch_v<32>(a, blocks, acc, grad_out, st);
        case 64: return launch_v<64>(a, blocks, acc, grad_out, st);
        case 128: return launch_v<128>(a, blocks, acc, grad_out, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
