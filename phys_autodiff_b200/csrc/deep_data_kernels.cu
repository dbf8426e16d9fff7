// The deep data-fit kernels; see deep_data_kernels.cuh for what they compute and deep_data_body.cuh for the kernel,
// k_deep_data_grad<H>, whose source k_deep_pair_grad (deep_pair_kernels.cu) shares.
#define DEEP_DATA_KERNEL k_deep_data_grad
#define DEEP_DATA_PAIRS false
#include "deep_data_body.cuh"

namespace physad {

namespace {

// one thread per entry: block partials summed in block order
__global__ void k_deep_data_reduce(const double* __restrict__ partials, int blocks, size_t P, double* grad, double* acc) {
    const size_t e = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= P + 1) return;
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += partials[size_t(b) * (P + 1) + e];
    if (e < P) grad[e] = s;
    else acc[0] = s;
}

template <int H>
int launch_t(const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    constexpr size_t smem = Geo<H>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(k_deep_data_grad<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return int(e);
    k_deep_data_grad<H><<<blocks, NT, smem, st>>>(*static_cast<const MlpConst<H>*>(mlp_const), a);
    if ((e = cudaGetLastError()) != cudaSuccess) return int(e);
    return deep_data_reduce(a.partials, blocks, grad_len(H, a.hidden_layers), grad, acc, st);
}

}  // namespace

int deep_data_reduce(const double* partials, int blocks, size_t P, double* grad, double* acc, cudaStream_t st) {
    k_deep_data_reduce<<<unsigned((P + 1 + 255) / 256), 256, 0, st>>>(partials, blocks, P, grad, acc);
    return int(cudaGetLastError());
}

size_t deep_data_ckpt_floats(int H, int hidden_layers) {
    (void)H;   // RB x H x ROWS = 8 x 16 x 192 for every width
    return size_t(hidden_layers) * Geo<32>::ACT;
}

int deep_data_blocks(int H, long long n_points, int max_blocks) {
    const int pts = H == 32 ? Geo<32>::NROW : (H == 64 ? Geo<64>::NROW : Geo<128>::NROW);
    const long long tiles = (n_points + pts - 1) / pts;
    return int(tiles < max_blocks ? (tiles > 0 ? tiles : 1) : max_blocks);
}

int deep_data_launch(int H, const void* mlp_const, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    switch (H) {
        case 32: return launch_t<32>(mlp_const, a, blocks, grad, acc, st);
        case 64: return launch_t<64>(mlp_const, a, blocks, grad, acc, st);
        case 128: return launch_t<128>(mlp_const, a, blocks, grad, acc, st);
    }
    return int(cudaErrorInvalidValue);
}

}  // namespace physad
