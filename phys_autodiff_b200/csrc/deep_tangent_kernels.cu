// The analytic deep loss and its closed loop on the grid; see deep_tangent_kernels.cuh for what they compute and
// deep_tangent_body.cuh for the kernel, k_deep_tangent<H, GRAD>.
#define DEEP_TANGENT_KERNEL k_deep_tangent
#define DEEP_TANGENT_POINTS false
#include "deep_tangent_body.cuh"

namespace physad {

namespace {

// one thread per entry: block partials [blocks][P + 2] summed in block order
__global__ void k_deep_tangent_reduce(const double* __restrict__ partials, int blocks, size_t P, double* grad, double* acc) {
    const size_t e = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= P + 2) return;
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += partials[size_t(b) * (P + 2) + e];
    if (e < P) grad[e] = s;
    else acc[e - P] = s;
}

template <int H, bool GRAD>
int launch_t(const DeepTangentArgs& a, int blocks, double* acc, double* grad, cudaStream_t st) {
    constexpr size_t smem = Geo<H, GRAD>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_deep_tangent<H, GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_deep_tangent<H, GRAD><<<blocks, NT, smem, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    return deep_tangent_reduce(a.partials, blocks, GRAD ? grad_len(H, a.hidden_layers) : 0, acc, grad, st);
}

}  // namespace

int deep_tangent_reduce(const double* partials, int blocks, size_t P, double* acc, double* grad, cudaStream_t st) {
    k_deep_tangent_reduce<<<unsigned((P + 2 + 255) / 256), 256, 0, st>>>(partials, blocks, P, grad, acc);
    return int(cudaGetLastError());
}

size_t deep_tangent_ckpt_floats(int hidden_layers) {
    return size_t(hidden_layers) * Geo<32, true>::ACT;   // RB x H x ROWS = 20480 for every width
}

int deep_tangent_blocks(int H, long long n_points, int max_blocks) {
    const int pts = H == 32 ? Geo<32, true>::PTS_TILE : (H == 64 ? Geo<64, true>::PTS_TILE : Geo<128, true>::PTS_TILE);
    const long long tiles = (n_points + pts - 1) / pts;
    return int(tiles < max_blocks ? (tiles > 0 ? tiles : 1) : max_blocks);
}

int deep_tangent_launch(int H, bool grad, const DeepTangentArgs& a, int blocks, double* acc, double* grad_out, cudaStream_t st) {
    switch (H) {
        case 32: return grad ? launch_t<32, true>(a, blocks, acc, grad_out, st) : launch_t<32, false>(a, blocks, acc, grad_out, st);
        case 64: return grad ? launch_t<64, true>(a, blocks, acc, grad_out, st) : launch_t<64, false>(a, blocks, acc, grad_out, st);
        case 128: return grad ? launch_t<128, true>(a, blocks, acc, grad_out, st) : launch_t<128, false>(a, blocks, acc, grad_out, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
