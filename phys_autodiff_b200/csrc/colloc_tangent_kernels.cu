// The analytic deep loss and its closed loop at caller-supplied points (collocation points); see deep_tangent_kernels.cuh
// for what they compute and deep_tangent_body.cuh for the kernel, k_colloc_tangent<H, GRAD>, whose source k_deep_tangent
// shares.  A translation unit of its own, so the grid kernels' object keeps exactly its six instantiations and the
// reduction.
#define DEEP_TANGENT_KERNEL k_colloc_tangent
#define DEEP_TANGENT_POINTS true
#include "deep_tangent_body.cuh"

namespace physad {

namespace {

template <int H, bool GRAD>
int launch_c(const DeepTangentArgs& a, int blocks, double* acc, double* grad, cudaStream_t st) {
    constexpr size_t smem = Geo<H, GRAD>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_colloc_tangent<H, GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_colloc_tangent<H, GRAD><<<blocks, NT, smem, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    return deep_tangent_reduce(a.partials, blocks, GRAD ? grad_len(H, a.hidden_layers) : 0, acc, grad, st);
}

}  // namespace

int colloc_tangent_launch(int H, bool grad, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st) {
    switch (H) {
        case 32: return grad ? launch_c<32, true>(a, blocks, acc, grad_out, st) : launch_c<32, false>(a, blocks, acc, grad_out, st);
        case 64: return grad ? launch_c<64, true>(a, blocks, acc, grad_out, st) : launch_c<64, false>(a, blocks, acc, grad_out, st);
        case 128: return grad ? launch_c<128, true>(a, blocks, acc, grad_out, st) : launch_c<128, false>(a, blocks, acc, grad_out, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
