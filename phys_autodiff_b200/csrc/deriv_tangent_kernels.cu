// The Jacobian of deep networks at caller-supplied points and the derivative-fit loss with its gradient (Neumann
// boundaries at points); see deep_tangent_kernels.cuh for what they compute and deep_tangent_body.cuh for the kernel,
// k_deriv_tangent<H, GRAD>, whose source k_deep_tangent and k_colloc_tangent share.  A translation unit of its own, so the
// other two objects keep exactly their instantiations.
#define DEEP_TANGENT_KERNEL k_deriv_tangent
#define DEEP_TANGENT_POINTS true
#define DEEP_TANGENT_DERIV true
#include "deep_tangent_body.cuh"

namespace physad {

namespace {

template <int H, bool GRAD>
int launch_d(const DeepTangentArgs& a, int blocks, double* acc, double* grad, cudaStream_t st) {
    constexpr size_t smem = Geo<H, GRAD>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_deriv_tangent<H, GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_deriv_tangent<H, GRAD><<<blocks, NT, smem, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    return GRAD ? deep_tangent_reduce(a.partials, blocks, grad_len(H, a.hidden_layers), acc, grad, st) : 0;
}

}  // namespace

int deriv_tangent_launch(int H, bool grad, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st) {
    switch (H) {
        case 32: return grad ? launch_d<32, true>(a, blocks, acc, grad_out, st) : launch_d<32, false>(a, blocks, acc, grad_out, st);
        case 64: return grad ? launch_d<64, true>(a, blocks, acc, grad_out, st) : launch_d<64, false>(a, blocks, acc, grad_out, st);
        case 128: return grad ? launch_d<128, true>(a, blocks, acc, grad_out, st) : launch_d<128, false>(a, blocks, acc, grad_out, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
