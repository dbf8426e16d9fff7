// C-ABI implementation (include/physad_b200.h): context, resident weights, launch geometry and
// the host-pointer staging wrappers.  All arithmetic lives in the kernels (*.cuh); this file only
// decides shapes, fills the kernel-parameter weight block and moves bytes.
#include "../../include/physad_b200.h"
#include "deep_data_kernels.cuh"
#include "deep_grad_kernels.cuh"
#include "deep_kernels.cuh"
#include "deep_tangent_kernels.cuh"
#include "deep_tc_kernels.cuh"
#include "dense_kernels.cuh"
#include "grad_kernels.cuh"
#include "stage_kernels.cuh"
#include "tangent_grad_kernels.cuh"
#include "tangent_kernels.cuh"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

using namespace physad;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(int(e_), std::string(#expr) + ": " + cudaGetErrorString(e_));              \
    } while (0)

}  // namespace

struct physad_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;  // used by the *_host entry points
    physad_mlp_config cfg{4, 0, 4, 1};
    bool has_weights = false;
    bool dev_weights_stale = true;
    std::vector<float> W1, b1, W2, b2;                             // host copy (feeds the parameter block)
    float *dW1 = nullptr, *db1 = nullptr, *dW2 = nullptr, *db2 = nullptr;  // device copy (generic MLP kernels)
    size_t dW_cap[4] = {0, 0, 0, 0};
    double2* partials = nullptr;
    size_t partials_cap = 0;
    unsigned int* ticket = nullptr;
    double* d_acc = nullptr;  // [2]
    double* h_acc = nullptr;  // pinned [2]
    // result record of the host-buffer fused calls: mapped pinned host memory the kernel's last block writes
    // directly (fused_loss.cuh: HostResult); the host polls `seq` instead of memcpy + stream sync
    HostResult* h_res = nullptr;        // host view
    HostResult* d_res = nullptr;        // device view of the same allocation
    unsigned long long res_seq = 0;     // last sequence number handed to a launch
    unsigned long long want_host_seq = 0;  // != 0: the next fused launch publishes into h_res with this seq
    unsigned int* d_status = nullptr;   // device word: 1 = an exchange timed out (sticky until physad_xchg_status reads it)
    unsigned long long* trace = nullptr;   // diagnostics: per-block timeline buffer of the next fused launches (device) or null
    int trace_blocks = 0;
    char* scratch = nullptr;  // device staging for *_host calls
    size_t scratch_cap = 0;
    // closed-loop gradient (physad_fused_loss_grad_*): fields + residuals workspace, block partials, result
    float* gws = nullptr;
    size_t gws_cap = 0;
    double* gpart = nullptr;
    size_t gpart_cap = 0;
    int grad_blocks_per_sm[3] = {0, 0, 0};   // HT = 32, 64, 128 on this device
    int tgrad_blocks_per_sm[3] = {0, 0, 0};  // the same for the tangent-loss gradient (physad_tangent_loss_grad_*)
    // deep closed loop (physad_deep_loss_grad_*): per-block activation checkpoints; the host forms' result [acc | grad]
    float* dckpt = nullptr;
    size_t dckpt_cap = 0;
    double* d_dgrad = nullptr;   // [P + 2]
    double* h_dgrad = nullptr;   // pinned, same size
    size_t d_dgrad_cap = 0, h_dgrad_cap = 0;
    uint64_t launches = 0;
    int fused_variant = 0;
    int exact_residuals = 0;  // 1: residual arithmetic in double exactly as the CPU reference; 0: fp32 with FMAs
    int advection = 0;        // 0: central differences (the reference); 1: first-order upwind advection (additive switch)
    // deeper MLPs (physad_set_weights_deep): hidden->hidden layers in the kernel's layout
    int deep_layers = 0;          // L (0 = not set)
    float *d_wh = nullptr, *d_bh = nullptr;
    size_t d_wh_cap = 0, d_bh_cap = 0;
    int deep_mode = 0;            // 0: strict fp32 on the CUDA cores; 1: hidden layers on tcgen05 (three-term bf16, deep_tc_kernels.cu)
    bool deep_tc_ok = false;      // the current deep weights have operand images
    uint8_t* d_wparts = nullptr;  // operand images of the hidden->hidden layers for mode 1 (null: shape not supported there)
    size_t d_wparts_cap = 0;
    // per-kernel launch facts on THIS device (opt-in shared memory set, resident blocks per SM): function
    // attributes are per device, so they are cached per context, not per process
    std::unordered_map<const void*, int> blocks_per_sm;
    // axis-coordinate tables cxs[nx] | cys[ny] | czs[nz] on the device, cached per (grid, norm)
    struct CoordTables {
        int key[5] = {0, 0, 0, 0, 0};  // nx, ny, nz, norm, valid
        float* dev = nullptr;
        size_t cap = 0;
    } tab;
    // launch plan of the fused kernel: coordinate tables + per-block work ranges, cached per geometry
    struct FusedPlan {
        int key[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // nx, ny, nz, z_begin, z_end, norm, TX, TY, slots, valid
        char* dev = nullptr;
        size_t cap = 0;
        const float *cxs = nullptr, *cys = nullptr, *czs = nullptr;
        const int* ranges = nullptr;
        int blocks = 0;
    } plan;
    // multi-GPU exchange through peer memory (physad_xchg_*)
    XSlot* xbuf = nullptr;                       // own buffer: [2][XCHG_MAX_RANKS] slots
    XSlot* xpeer[XCHG_MAX_RANKS] = {};           // every rank's buffer as mapped in this process
    int xrank = 0, xworld = 1;
    unsigned long long xepoch = 0;
};

namespace {

// Grow the context buffer p of cap elements to at least n (device memory, or pinned host memory).  It never shrinks and
// keeps no contents: every caller refills the buffer.  The old buffer is freed before the new one is allocated, so the peak
// does not double, and a failed allocation leaves (nullptr, 0) so that the next call tries again.
template <class T>
int grow(T*& p, size_t& cap, size_t n, bool pinned = false) {
    if (n <= cap) return 0;
    if (p) CU(pinned ? cudaFreeHost(p) : cudaFree(p));
    p = nullptr;
    cap = 0;
    void* q = nullptr;
    CU(pinned ? cudaMallocHost(&q, n * sizeof(T)) : cudaMalloc(&q, n * sizeof(T)));
    p = static_cast<T*>(q);
    cap = n;
    return 0;
}

int ensure_partials(physad_ctx* c, size_t blocks) { return grow(c->partials, c->partials_cap, blocks); }
int ensure_scratch(physad_ctx* c, size_t bytes) { return grow(c->scratch, c->scratch_cap, bytes); }
int ensure_grad_partials(physad_ctx* c, size_t doubles) { return grow(c->gpart, c->gpart_cap, doubles); }

int check_grid(const physad_grid* g) {
    if (!g) return fail(PHYSAD_E_INVALID, "grid is null");
    if (g->nx <= 0 || g->ny <= 0 || g->nz <= 0) return fail(PHYSAD_E_INVALID, "grid extents must be positive");
    if (size_t(g->nx) * g->ny * g->nz >= (size_t(1) << 31))
        return fail(PHYSAD_E_UNSUPPORTED, "N >= 2^31 (the reference indexes with int, src/phys_cuda_fused.cu:187)");
    return 0;
}

int check_slab(const physad_grid* g, const physad_slab* s, physad_slab* out) {
    physad_slab r{0, g->nz};
    if (s) r = *s;
    if (r.z_begin < 0 || r.z_end > g->nz || r.z_begin > r.z_end) return fail(PHYSAD_E_INVALID, "slab outside the grid");
    *out = r;
    return 0;
}

// float(1 / (2 h)) with the quotient formed in double as the CPU reference does (src/phys_cpu.cpp:38-41)
float inv2(float h) { return float(1.0 / (2.0 * double(h))); }
double inv2d(float h) { return 1.0 / (2.0 * double(h)); }  // exactly src/phys_cpu.cpp:38-41

int template_h(int H) { return H <= 32 ? 32 : (H <= 64 ? 64 : (H <= 128 ? 128 : 0)); }

// Fill the kernel-parameter weight block.  Hidden units beyond cfg.H are zero records: they
// contribute act = relu(0) = 0 and products 0, which leave every accumulator unchanged.
template <int H>
void fill_const(const physad_ctx* c, const float tcoord[3], MlpConst<H>& k) {
    const int h_rt = c->cfg.H;
    auto W1 = [&](int h, int col) { return h < h_rt ? c->W1[size_t(h) * 4 + col] : 0.f; };
    auto B1 = [&](int h) { return h < h_rt ? c->b1[h] : 0.f; };
    auto W2 = [&](int o, int h) { return h < h_rt ? c->W2[size_t(o) * h_rt + h] : 0.f; };
    // separately rounded fp32 product W1[h,3]*t (volatile: nothing wider, nothing fused)
    auto PT = [&](int h, int s) { volatile float p = W1(h, 3) * tcoord[s]; return float(p); };
    for (int q = 0; q < H / 2; ++q) {
        const int h0 = 2 * q, h1 = 2 * q + 1;
        k.b1p[q] = make_float2(B1(h0), B1(h1));
        k.w0s[q] = make_float2(W1(h1, 0), W1(h0, 0));
        k.w1s[q] = make_float2(W1(h1, 1), W1(h0, 1));
        k.w2s[q] = make_float2(W1(h1, 2), W1(h0, 2));
        k.ptm[q] = make_float2(PT(h0, 0), PT(h1, 0));
        k.pt0[q] = make_float2(PT(h0, 1), PT(h1, 1));
        k.ptp[q] = make_float2(PT(h0, 2), PT(h1, 2));
    }
    for (int h = 0; h < H; ++h) k.w2[h] = make_float4(W2(1, h), W2(0, h), W2(3, h), W2(2, h));
    k.b2 = make_float4(c->b2[0], c->b2[1], c->b2[2], c->b2[3]);
}

// 4th MLP input for a time value (reference src/mlp_grid.cpp:38)
float time_coord(float t, int norm) { return norm == 1 ? t : (t + 0.5f); }

// The one-hidden-layer entry points read only the first and the last layer of the context's weights.  After
// physad_set_weights_deep with L > 1 that pair is not the network the caller set, so they refuse it instead of
// evaluating 4 -> H -> 4 with the hidden -> hidden layers dropped.
int need_one_layer(const physad_ctx* c, const char* what, const char* deep_twin) {
    if (c->deep_layers <= 1) return 0;
    std::string msg = std::string(what) + ": one-hidden-layer entry point, but the context holds a network of " +
                      std::to_string(c->deep_layers) + " hidden layers (physad_set_weights_deep)";
    if (deep_twin) msg += std::string("; use ") + deep_twin;
    return fail(PHYSAD_E_UNSUPPORTED, msg);
}

int need_4x4(const physad_ctx* c, const char* what, const char* deep_twin) {
    if (!c->has_weights) return fail(PHYSAD_E_NOWEIGHTS, std::string(what) + ": no weights set");
    if (int rc = need_one_layer(c, what, deep_twin)) return rc;
    if (c->cfg.In != 4 || c->cfg.Out != 4)
        return fail(PHYSAD_E_UNSUPPORTED, std::string(what) + ": grid paths need In = Out = 4 (src/mlp_grid.cpp:69-80)");
    if (template_h(c->cfg.H) == 0) return fail(PHYSAD_E_UNSUPPORTED, std::string(what) + ": H > 128 not built");
    return 0;
}

// ---- fused kernel launch -----------------------------------------------------------------
// Axis coordinate exactly as the reference forms it (src/mlp_grid.cpp:25-29; this TU is compiled
// with -ffp-contract=off): u = float(i)/float(n-1), MinusOneToOne -> 2u-1.
float host_axis_coord(int i, int n, bool m1p1) {
    if (n <= 1) return 0.0f;
    volatile float u = float(i) / float(n - 1);
    volatile float two_u = 2.f * u;
    return m1p1 ? two_u - 1.f : float(u);
}

// Device tables of the axis coordinates of every x, y and z index (a few KB), so kernels neither divide
// nor recompute them per point.  Rebuilt only when the grid extents or the normalisation change.
int ensure_coord_tables(physad_ctx* c, const physad_grid* g, cudaStream_t st) {
    const int key[5] = {g->nx, g->ny, g->nz, c->cfg.norm, 1};
    auto& t = c->tab;
    if (std::memcmp(key, t.key, sizeof(key)) == 0) return 0;
    const bool m1p1 = c->cfg.norm == 1;
    const size_t nf = size_t(g->nx) + g->ny + g->nz;
    std::vector<float> host(nf);
    for (int i = 0; i < g->nx; ++i) host[i] = host_axis_coord(i, g->nx, m1p1);
    for (int i = 0; i < g->ny; ++i) host[g->nx + i] = host_axis_coord(i, g->ny, m1p1);
    for (int i = 0; i < g->nz; ++i) host[g->nx + g->ny + i] = host_axis_coord(i, g->nz, m1p1);
    if (int rc = grow(t.dev, t.cap, nf)) return rc;
    // rare path: copy on the CONSUMING stream and wait, so the first kernel after a geometry change cannot read
    // stale tables (a NULL-stream copy is not ordered against a cudaStreamNonBlocking stream) and the pageable
    // staging vector may die at the end of this scope
    CU(cudaMemcpyAsync(t.dev, host.data(), nf * sizeof(float), cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    std::memcpy(t.key, key, sizeof(key));
    return 0;
}

// Split the tile-plane sequence (tiles x nzl planes, tile-major) into at most `slots` contiguous ranges
// of equal COST, where a range pays `seg_cost` extra for every z-segment it starts (its two time-t-only
// halo planes + prologue).  Greedy fill under a cost cap, cap found by bisection.
std::vector<int> balanced_ranges(int tiles, int nzl, long long slots, double seg_cost) {
    auto fill = [&](double cap, std::vector<int>* out) {
        long long blocks = 0;
        double cur = 0.0;
        bool open = false;
        if (out) { out->clear(); out->push_back(0); }
        for (int t = 0; t < tiles; ++t) {
            int rem = nzl;
            while (rem > 0) {
                const double space = cap - cur - seg_cost;
                if (space < 1.0 && open) {  // cannot start a segment here: close the block
                    ++blocks; cur = 0.0; open = false;
                    if (out) out->push_back(t * nzl + (nzl - rem));
                    continue;
                }
                const int take = std::max(1, std::min(rem, int(space)));
                cur += seg_cost + take;
                rem -= take;
                open = true;
                if (cur + seg_cost + 1.0 > cap) {
                    ++blocks; cur = 0.0; open = false;
                    if (out) out->push_back(t * nzl + (nzl - rem));
                }
            }
        }
        if (open) { ++blocks; if (out) out->push_back(tiles * nzl); }
        return blocks;
    };
    double lo = 1.0 + seg_cost, hi = double(tiles) * (nzl + seg_cost) + 1.0;
    for (int it = 0; it < 60; ++it) {
        const double mid = 0.5 * (lo + hi);
        if (fill(mid, nullptr) <= slots) hi = mid; else lo = mid;
    }
    std::vector<int> r;
    fill(hi, &r);
    return r;
}

int build_fused_plan(physad_ctx* c, const physad_grid* g, const physad_slab& s, int TX, int TY, long long slots,
                     cudaStream_t st) {
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    auto& p = c->plan;
    p.cxs = c->tab.dev;
    p.cys = p.cxs + g->nx;
    p.czs = p.cys + g->ny;
    const int key[10] = {g->nx, g->ny, g->nz, s.z_begin, s.z_end, c->cfg.norm, TX, TY, int(slots), 1};
    if (std::memcmp(key, p.key, sizeof(key)) == 0) return 0;
    const int tiles = ((g->nx + TX - 1) / TX) * ((g->ny + TY - 1) / TY), nzl = s.z_end - s.z_begin;
    const long long want = std::min<long long>(slots, (long long)tiles * nzl);
    const std::vector<int> ranges = balanced_ranges(tiles, nzl, want, 0.9);
    const size_t bytes = ranges.size() * sizeof(int);
    if (int rc = grow(p.dev, p.cap, bytes)) return rc;
    CU(cudaMemcpyAsync(p.dev, ranges.data(), bytes, cudaMemcpyHostToDevice, st));   // same ordering rule as the coordinate tables
    CU(cudaStreamSynchronize(st));
    p.ranges = reinterpret_cast<const int*>(p.dev);
    p.blocks = int(ranges.size()) - 1;
    std::memcpy(p.key, key, sizeof(key));
    return 0;
}

template <int H, int P, int TYB, int UNROLL, int MINB, bool PACKED, bool SPLITBAR, bool DPRES>
int launch_fused_d(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], bool xchg, double* acc,
                   float* const R[4], cudaStream_t st, int blocks_per_sm_cap = 0) {
    constexpr int TX = 32, TY = TYB * P;
    auto kern = k_fused_mlp_phys_loss<H, P, TYB, UNROLL, MINB, PACKED, SPLITBAR, DPRES>;
    const size_t smem = size_t(4) * 4 * (TX + 2) * (TY + 2) * sizeof(float);
    // per-kernel launch facts, queried once per context (this sits on the per-step host path)
    static const long long env_blocks = getenv("PHYSAD_FUSED_BLOCKS") ? atoll(getenv("PHYSAD_FUSED_BLOCKS")) : 0;  // tuning aid
    int& per_sm = c->blocks_per_sm[reinterpret_cast<const void*>(kern)];
    if (per_sm == 0) {
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        int q = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, 32 * TYB, smem));
        if (q < 1) return fail(PHYSAD_E_UNSUPPORTED, "fused kernel does not fit on an SM");
        per_sm = q;
    }
    const int tiles_x = (g->nx + TX - 1) / TX, tiles_y = (g->ny + TY - 1) / TY;
    // persistent grid: one block per resident slot, each owning an equal-cost share of the tile-planes
    const int bps = blocks_per_sm_cap > 0 ? std::min(per_sm, blocks_per_sm_cap) : per_sm;
    const long long slots = env_blocks > 0 ? env_blocks : (long long)bps * c->sm_count;
    if (int rc = build_fused_plan(c, g, s, TX, TY, slots, st)) return rc;
    const long long blocks = c->plan.blocks;
    FusedArgs a{};
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz;
    a.z_begin = s.z_begin; a.z_end = s.z_end;
    a.tiles_x = tiles_x; a.tiles_y = tiles_y;
    a.cxs = c->plan.cxs; a.cys = c->plan.cys; a.czs = c->plan.czs; a.ranges = c->plan.ranges;
    a.m1p1 = c->cfg.norm == 1; a.periodic = g->periodic != 0;
    a.inv2dt = inv2(g->dt); a.inv2hx = inv2(g->hx); a.inv2hy = inv2(g->hy); a.inv2hz = inv2(g->hz);
    a.inv2dt_d = inv2d(g->dt); a.inv2hx_d = inv2d(g->hx); a.inv2hy_d = inv2d(g->hy); a.inv2hz_d = inv2d(g->hz);
    if (int rc = ensure_partials(c, size_t(blocks))) return rc;
    a.partials = c->partials; a.ticket = c->ticket; a.acc_out = acc;
    for (int k = 0; k < 4; ++k) a.R[k] = R[k];
    if (xchg) {
        a.x.rank = c->xrank; a.x.world = c->xworld; a.x.epoch = c->xepoch + 1;
        for (int p = 0; p < XCHG_MAX_RANKS; ++p) a.x.peer[p] = c->xpeer[p];
    }
    a.status = c->d_status;
    if (c->want_host_seq) { a.host_res = c->d_res; a.host_seq = c->want_host_seq; }
    if (c->trace && blocks <= c->trace_blocks) a.trace = c->trace;
    MlpConst<H> k;
    fill_const<H>(c, tc, k);
    kern<<<unsigned(blocks), 32 * TYB, smem, st>>>(k, a);
    CU(cudaGetLastError());
    c->launches++;
    if (xchg) c->xepoch++;   // only a launch that went out consumes an epoch (every rank makes the same calls)
    return 0;
}

// fp32-residual launch of a given geometry (all tuning variants)
template <int H, int P, int TYB, int UNROLL, int MINB, bool PACKED, bool SPLITBAR = false>
int launch_fused_t(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], bool xchg, double* acc,
                   float* const R[4], cudaStream_t st, int blocks_per_sm_cap = 0) {
    return launch_fused_d<H, P, TYB, UNROLL, MINB, PACKED, SPLITBAR, false>(c, g, s, tc, xchg, acc, R, st, blocks_per_sm_cap);
}

// The default geometry: one 512-thread block/SM on 32x64 tiles; for small slabs (multi-GPU strong scaling: a block's
// share is only a few planes, and every z-segment costs ~1.15 plane-steps of halo + prologue) one 256-thread
// block/SM on 32x32 tiles, which halves the number of z-segments (measured 0.1626 vs 0.1668 ms on 256x256x32).
template <int H, bool DPRES>
int launch_fused_default(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], bool xchg,
                         double* acc, float* const R[4], cudaStream_t st) {
    const long long tile_planes = (long long)((g->nx + 31) / 32) * ((g->ny + 63) / 64) * (s.z_end - s.z_begin);
    if (tile_planes < 12LL * c->sm_count)
        return launch_fused_d<H, 4, 8, 2, 2, true, true, DPRES>(c, g, s, tc, xchg, acc, R, st, 1);
    return launch_fused_d<H, 4, 16, 2, 1, true, true, DPRES>(c, g, s, tc, xchg, acc, R, st, 0);
}

template <int H>
int launch_fused_h(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], bool dt, double* acc,
                   float* const R[4], cudaStream_t st) {
    // exact (double) residual arithmetic is built for the default geometry only
    if (c->exact_residuals) return launch_fused_default<H, true>(c, g, s, tc, dt, acc, R, st);
    // <H, P columns/thread, warps/block, unroll (pairs of hidden units), min blocks/SM, packed, split barrier>
    switch (c->fused_variant) {
        default:
        case 0: return launch_fused_default<H, false>(c, g, s, tc, dt, acc, R, st);
        case 1: return launch_fused_t<H, 4, 8, 2, 2, true, true>(c, g, s, tc, dt, acc, R, st);    // tile 32x32, 2 x 256 threads/SM
        case 2: return launch_fused_t<H, 4, 16, 2, 1, true, false>(c, g, s, tc, dt, acc, R, st);  // variant 0 with __syncthreads
        case 3: return launch_fused_t<H, 4, 8, 2, 1, false, false>(c, g, s, tc, dt, acc, R, st);  // scalar FMUL/FADD cross-check
        case 4: return launch_fused_t<H, 2, 16, 4, 1, true, true>(c, g, s, tc, dt, acc, R, st);   // tile 32x32, 1 x 512
        case 5: return launch_fused_t<H, 1, 8, 4, 4, true, false>(c, g, s, tc, dt, acc, R, st);   // tile 32x8
        case 6: return launch_fused_t<H, 2, 8, 2, 3, true, true>(c, g, s, tc, dt, acc, R, st);    // tile 32x16, 3 x 256
        case 7: return launch_fused_t<H, 4, 8, 2, 2, true, true>(c, g, s, tc, dt, acc, R, st, 1); // tile 32x32, ONE 256-thread block/SM
    }
}

int launch_fused(physad_ctx* c, const physad_grid* g, const physad_slab& s, float t, float dt, double* acc,
                 float* const R[4], cudaStream_t st, bool xchg = false) {
    if (c->advection != 0)
        return fail(PHYSAD_E_UNSUPPORTED, "fused_loss: the fused kernel implements the reference's central scheme only; "
                                          "upwind advection runs stage-wise (generate_fields + phys_loss)");
    if (xchg && (c->xworld <= 1 || !c->xbuf))
        return fail(PHYSAD_E_INVALID, "fused_loss_allreduce: call physad_xchg_connect first");
    if (s.z_end == s.z_begin) {  // empty slab: the sum over nothing (still takes part in the exchange)
        XchgArgs x{};
        if (xchg) {
            x.rank = c->xrank; x.world = c->xworld; x.epoch = c->xepoch + 1;
            for (int p = 0; p < XCHG_MAX_RANKS; ++p) x.peer[p] = c->xpeer[p];
        }
        k_xchg_only<<<1, 32, 0, st>>>(x, acc, c->want_host_seq ? c->d_res : nullptr, c->want_host_seq, c->d_status);
        CU(cudaGetLastError());
        c->launches++;
        if (xchg) c->xepoch++;
        return 0;
    }
    const float ts[3] = {t - dt, t, t + dt};  // as src/mlp_grid.cpp:87-89
    const float tc[3] = {time_coord(ts[0], c->cfg.norm), time_coord(ts[1], c->cfg.norm), time_coord(ts[2], c->cfg.norm)};
    switch (template_h(c->cfg.H)) {
        case 32: return launch_fused_h<32>(c, g, s, tc, xchg, acc, R, st);
        case 64: return launch_fused_h<64>(c, g, s, tc, xchg, acc, R, st);
        case 128: return launch_fused_h<128>(c, g, s, tc, xchg, acc, R, st);
    }
    return fail(PHYSAD_E_UNSUPPORTED, "H > 128 not built");
}

// ---- MLP over the grid ---------------------------------------------------------------------
template <int H, bool FIELDS>
int launch_grid_t(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], GridInferArgs a,
                  cudaStream_t st, int dtype = PHYSAD_F32) {
    const int nzl = s.z_end - s.z_begin;
    if (nzl == 0) return 0;
    // a block covers 32 rows: gridDim.y caps ny at 65535 * 32
    if ((g->ny + 31) / 32 > 65535) return fail(PHYSAD_E_UNSUPPORTED, "grid MLP kernels: ny > 2097120");
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    a.cxs = c->tab.dev; a.cys = a.cxs + g->nx; a.czs = a.cys + g->ny;
    MlpConst<H> k;
    fill_const<H>(c, tc, k);
    // one plane per blockIdx.z, so more than 65535 planes go out in bands; the kernel indexes its outputs from the
    // band's first plane, and the u arrays keep the channel stride of the whole slab
    const size_t pln = size_t(g->nx) * g->ny;
    const size_t esz = (FIELDS && dtype != PHYSAD_F32) ? 2 : sizeof(float);   // bytes per stored field element
    if (a.cstride == 0) a.cstride = size_t(nzl) * pln;
    for (int z0 = s.z_begin; z0 < s.z_end; z0 += 65535) {
        const int nb = std::min(65535, s.z_end - z0);
        const size_t off = size_t(z0 - s.z_begin) * pln;
        GridInferArgs b = a;
        b.z_begin = z0; b.z_end = z0 + nb;
        if (FIELDS) {
            for (int q = 0; q < 3; ++q) {
                b.sigma[q] = reinterpret_cast<float*>(reinterpret_cast<char*>(a.sigma[q]) + off * esz);
                b.u[q] = reinterpret_cast<float*>(reinterpret_cast<char*>(a.u[q]) + off * esz);
            }
        } else {
            b.out_aos = a.out_aos + off;
        }
        const dim3 grid(unsigned((g->nx + 31) / 32), unsigned((g->ny + 31) / 32), unsigned(nb));
        if (FIELDS && dtype == PHYSAD_F16) k_mlp_grid<H, FIELDS, 2, __half><<<grid, 256, 0, st>>>(k, b);
        else if (FIELDS && dtype == PHYSAD_BF16) k_mlp_grid<H, FIELDS, 2, __nv_bfloat16><<<grid, 256, 0, st>>>(k, b);
        else k_mlp_grid<H, FIELDS, 2><<<grid, 256, 0, st>>>(k, b);
        c->launches++;
        CU(cudaGetLastError());
    }
    return 0;
}

template <bool FIELDS>
int launch_grid(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], GridInferArgs a,
                cudaStream_t st, int dtype = PHYSAD_F32) {
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz;
    a.z_begin = s.z_begin; a.z_end = s.z_end;
    a.m1p1 = c->cfg.norm == 1;
    switch (template_h(c->cfg.H)) {
        case 32: return launch_grid_t<32, FIELDS>(c, g, s, tc, a, st, dtype);
        case 64: return launch_grid_t<64, FIELDS>(c, g, s, tc, a, st, dtype);
        case 128: return launch_grid_t<128, FIELDS>(c, g, s, tc, a, st, dtype);
    }
    return fail(PHYSAD_E_UNSUPPORTED, "H > 128 not built");
}

// ---- physics on supplied fields --------------------------------------------------------------
template <bool WRITE_R, bool REDUCE, bool SCALE>
int launch_phys(physad_ctx* c, const physad_grid* g_in, PhysArgs a, cudaStream_t st, int slab_planes = -1, int dtype = PHYSAD_F32) {
    // slab mode: the arrays hold `slab_planes` planes and the z neighbours outside them come from a.halo_lo/hi
    physad_grid gl = *g_in;
    if (slab_planes >= 0) gl.nz = slab_planes;
    const physad_grid* g = &gl;
    if (g->nz == 0) {
        if (REDUCE) CU(cudaMemsetAsync(a.acc_out, 0, 2 * sizeof(double), st));
        return 0;
    }
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz; a.periodic = g->periodic != 0;
    a.inv2dt = inv2(g->dt); a.inv2hx = inv2(g->hx); a.inv2hy = inv2(g->hy); a.inv2hz = inv2(g->hz);
    a.inv2dt_d = inv2d(g->dt); a.inv2hx_d = inv2d(g->hx); a.inv2hy_d = inv2d(g->hy); a.inv2hz_d = inv2d(g->hz);
    a.inv1hx_d = 1.0 / double(g->hx); a.inv1hy_d = 1.0 / double(g->hy); a.inv1hz_d = 1.0 / double(g->hz);
    a.inv1hx = float(a.inv1hx_d); a.inv1hy = float(a.inv1hy_d); a.inv1hz = float(a.inv1hz_d);
    const bool upwind = c->advection == 1;
    // 128-bit form when rows are quad-aligned and wide enough to fill the 64-quad blocks reasonably (central scheme only)
    static const bool no_v4 = getenv("PHYSAD_NO_V4") != nullptr;  // tuning aid
    bool v4 = !upwind && !no_v4 && g->nx % 4 == 0 && (g->nx >= 128 || dtype != PHYSAD_F32);
    const void* ptrs[12] = {a.s_m, a.s_0, a.s_p, a.u_m, a.u_0, a.u_p, a.R[0], a.R[1], a.R[2], a.R[3], a.halo_lo, a.halo_hi};
    for (int k = 0; k < 12; ++k) v4 = v4 && (uintptr_t(ptrs[k]) % ((dtype != PHYSAD_F32 && (k < 6 || k >= 10)) ? 8 : 16) == 0);
    v4 = v4 && (size_t(g->nx) * g->ny * g->nz) % 4 == 0;  // channel stride of the u arrays
    // the v4 grid has one block row per 2 rows (gridDim.y <= 65535): fp32 fields beyond that take the scalar kernel
    const bool v4_rows = (g->ny + V4_THREADS / 64 - 1) / (V4_THREADS / 64) <= 65535;
    if (dtype == PHYSAD_F32) v4 = v4 && v4_rows;
    if (dtype != PHYSAD_F32 && (!v4 || SCALE || c->exact_residuals))
        return fail(PHYSAD_E_UNSUPPORTED, "16-bit fields: need nx % 4 == 0, 8-byte aligned arrays, the central scheme and fp32 residual arithmetic");
    if (v4) {
        const unsigned tx = unsigned((g->nx + 255) / 256), ty = unsigned((g->ny + V4_THREADS / 64 - 1) / (V4_THREADS / 64));
        if (ty > 65535u) return fail(PHYSAD_E_UNSUPPORTED, "phys kernels: 16-bit fields need ny <= 131070");
        const long long want = (long long)c->sm_count * 8;
        long long nch = std::max(1LL, std::min<long long>(g->nz, (want + (long long)tx * ty - 1) / ((long long)tx * ty)));
        a.zc = int((g->nz + nch - 1) / nch);
        nch = (g->nz + a.zc - 1) / a.zc;
        if (nch > 65535) { a.zc = (g->nz + 65534) / 65535; nch = (g->nz + a.zc - 1) / a.zc; }
        const dim3 grid(tx, ty, unsigned(nch));
        if (REDUCE) {
            if (int rc = ensure_partials(c, size_t(tx) * ty * nch)) return rc;
            a.partials = c->partials; a.ticket = c->ticket;
        }
        if constexpr (!SCALE) {
            if (dtype == PHYSAD_F16) k_phys_residual_v4<WRITE_R, REDUCE, SCALE, false, __half><<<grid, V4_THREADS, 0, st>>>(a);
            else if (dtype == PHYSAD_BF16) k_phys_residual_v4<WRITE_R, REDUCE, SCALE, false, __nv_bfloat16><<<grid, V4_THREADS, 0, st>>>(a);
        }
        if (dtype != PHYSAD_F32) { }
        else if (c->exact_residuals) k_phys_residual_v4<WRITE_R, REDUCE, SCALE, true><<<grid, V4_THREADS, 0, st>>>(a);
        else k_phys_residual_v4<WRITE_R, REDUCE, SCALE, false><<<grid, V4_THREADS, 0, st>>>(a);
        c->launches++;
        CU(cudaGetLastError());
        return 0;
    }
    // 32 x 8 column tiles, each marching a z chunk; enough chunks for ~16 blocks per SM
    const unsigned tx = unsigned((g->nx + 31) / 32), ty = unsigned((g->ny + 7) / 8);
    if (ty > 65535u) return fail(PHYSAD_E_UNSUPPORTED, "phys kernels: ny > 524280");
    const long long want = (long long)c->sm_count * 16;
    long long nch = std::max(1LL, std::min<long long>(g->nz, (want + (long long)tx * ty - 1) / ((long long)tx * ty)));
    a.zc = int((g->nz + nch - 1) / nch);
    nch = (g->nz + a.zc - 1) / a.zc;
    if (nch > 65535) { a.zc = (g->nz + 65534) / 65535; nch = (g->nz + a.zc - 1) / a.zc; }
    const dim3 grid(tx, ty, unsigned(nch));
    if (REDUCE) {
        if (int rc = ensure_partials(c, size_t(tx) * ty * nch)) return rc;
        a.partials = c->partials; a.ticket = c->ticket;
    }
    if (upwind) {
        if (c->exact_residuals) k_phys_residual<WRITE_R, REDUCE, SCALE, true, true><<<grid, 256, 0, st>>>(a);
        else k_phys_residual<WRITE_R, REDUCE, SCALE, false, true><<<grid, 256, 0, st>>>(a);
    } else if (c->exact_residuals) k_phys_residual<WRITE_R, REDUCE, SCALE, true><<<grid, 256, 0, st>>>(a);
    else k_phys_residual<WRITE_R, REDUCE, SCALE, false><<<grid, 256, 0, st>>>(a);
    c->launches++;
    CU(cudaGetLastError());
    return 0;
}

PhysArgs phys_args(const float* s_m, const float* s_0, const float* s_p, const float* u_m, const float* u_0,
                   const float* u_p, float* r0, float* r1, float* r2, float* r3) {
    PhysArgs a{};
    a.s_m = s_m; a.s_0 = s_0; a.s_p = s_p; a.u_m = u_m; a.u_0 = u_0; a.u_p = u_p;
    a.R[0] = r0; a.R[1] = r1; a.R[2] = r2; a.R[3] = r3;
    return a;
}

// VJP scales formed in fp32 exactly as src/phys_cpu.cpp:162-163
void vjp_scales(const physad_grid* g, const physad_phys_weights* w, float* ss, float* su) {
    const size_t N = size_t(g->nx) * g->ny * g->nz;
    *ss = 2.f * w->w_sigma / float(N);
    *su = 2.f * w->w_u / float(N);
}

// dc/dx of the three space inputs of a grid: a coordinate c = norm(i / (n - 1)) sampled at x = i h has dc/dx = f / ((n-1) h),
// f = 2 for MinusOneToOne (norm 1), 1 for ZeroToOne, and 0 for an extent of 1
void input_scales(const physad_grid* g, int norm, float s[3]) {
    const double f = norm == 1 ? 2.0 : 1.0;
    s[0] = g->nx > 1 ? float(f / (double(g->nx - 1) * double(g->hx))) : 0.f;
    s[1] = g->ny > 1 ? float(f / (double(g->ny - 1) * double(g->hy))) : 0.f;
    s[2] = g->nz > 1 ? float(f / (double(g->nz - 1) * double(g->hz))) : 0.f;
}

int check_residual_outputs(const float* Rs, const float* Rx, const float* Ry, const float* Rz, const char* what) {
    const bool any = Rs || Rx || Ry || Rz, all = Rs && Rx && Ry && Rz;
    if (any && !all) return fail(PHYSAD_E_INVALID, std::string(what) + ": residual outputs must be all set or all null");
    return 0;
}

// The result of an empty slab or shard: nacc zero sums in acc and, if grad is set, a zero gradient of P entries
int zero_result(double* acc, int nacc, double* grad, size_t P, cudaStream_t st) {
    if (nacc) CU(cudaMemsetAsync(acc, 0, nacc * sizeof(double), st));
    if (grad) CU(cudaMemsetAsync(grad, 0, P * sizeof(double), st));
    return 0;
}

// One array of a host-pointer call, staged in the context's scratch: `up` is uploaded before the device call, `down`
// downloaded after it; either may be null (an input only, an output only, an output the caller did not ask for, or
// workspace).  `dev` is the array's place in scratch.
struct Staged {
    const void* up;
    void* down;
    size_t bytes;
    float* dev = nullptr;
};

// Lay the arrays out in scratch, each at a 256-byte aligned offset, and upload the inputs on c->stream.
template <size_t K>
int stage_in(physad_ctx* c, Staged (&a)[K]) {
    size_t off[K + 1] = {0};
    for (size_t k = 0; k < K; ++k) off[k + 1] = off[k] + ((a[k].bytes + 255) & ~size_t(255));
    if (int rc = grow(c->scratch, c->scratch_cap, off[K])) return rc;
    for (size_t k = 0; k < K; ++k) {
        a[k].dev = reinterpret_cast<float*>(c->scratch + off[k]);
        if (a[k].up && a[k].bytes) CU(cudaMemcpyAsync(a[k].dev, a[k].up, a[k].bytes, cudaMemcpyHostToDevice, c->stream));
    }
    return 0;
}

// After the device call: download the outputs and synchronise c->stream once.
template <size_t K>
int stage_out(physad_ctx* c, const Staged (&a)[K]) {
    for (const Staged& s : a)
        if (s.down && s.bytes) CU(cudaMemcpyAsync(s.down, s.dev, s.bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

}  // namespace

namespace {
int launch_grad(physad_ctx* c, int HT, const GradArgs& a, float4* adj, size_t chunks, cudaStream_t st) {
    int& bps = c->grad_blocks_per_sm[HT == 32 ? 0 : (HT == 64 ? 1 : 2)];
    if (!bps) {
        CU(cudaError_t(grad_blocks_per_sm(HT, &bps)));
        if (bps < 1) return fail(PHYSAD_E_UNSUPPORTED, "fused_loss_grad: kernel does not fit an SM");
    }
    const size_t blocks = std::max<size_t>(1, std::min<size_t>(chunks, size_t(c->sm_count) * bps));
    if (int rc = ensure_grad_partials(c, blocks * (GRAD_NACC * HT + 6))) return rc;
    GradArgs k = a;
    k.partials = c->gpart;
    c->launches += 2;
    CU(cudaError_t(adjoint_launch(k, adj, st)));
    CU(cudaError_t(grad_launch(HT, k, adj, unsigned(blocks), st)));
    return 0;
}
}  // namespace

namespace {
int upload_weights_if_stale(physad_ctx* c, cudaStream_t st) {
    if (!c->dev_weights_stale) return 0;
    std::vector<float>* host[4] = {&c->W1, &c->b1, &c->W2, &c->b2};
    float** dev[4] = {&c->dW1, &c->db1, &c->dW2, &c->db2};
    for (int k = 0; k < 4; ++k) {
        const size_t n = host[k]->size();
        if (int rc = grow(*dev[k], c->dW_cap[k], n)) return rc;
        // pageable source: the copy is staged before the call returns, so the host vector may change afterwards
        CU(cudaMemcpyAsync(*dev[k], host[k]->data(), n * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    c->dev_weights_stale = false;
    return 0;
}
}  // namespace

namespace {
template <int H, bool FIELDS>
int launch_deep(physad_ctx* c, const physad_grid* g, const physad_slab& s, const float tc[3], DeepArgs a, cudaStream_t st) {
    const int nzl = s.z_end - s.z_begin;
    if (nzl == 0) return 0;
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz; a.z_begin = s.z_begin; a.z_end = s.z_end;
    a.hidden_layers = c->deep_layers;
    a.cxs = c->tab.dev; a.cys = a.cxs + g->nx; a.czs = a.cys + g->ny;
    a.wh = c->d_wh; a.bh = c->d_bh;
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    a.W1 = c->dW1; a.b1 = c->db1;
    for (int k3 = 0; k3 < 3; ++k3) a.tc[k3] = tc[k3];
    MlpConst<H> k;
    fill_const<H>(c, tc, k);
    if (c->deep_mode == 1) {
        if (!deep_tc_supported(H, c->deep_layers) || !c->deep_tc_ok)
            return fail(PHYSAD_E_UNSUPPORTED, "deep fast mode: needs at least 2 hidden layers (the tensor cores only take the "
                                              "hidden -> hidden contractions)");
        CU(cudaError_t(deep_tc_launch(H, FIELDS, &k, a, c->d_wparts, c->sm_count, st)));
        c->launches++;
        return 0;
    }
    // persistent grid: one 256-thread block per SM, tiles of 64..768 points handed out round-robin (deep_kernels.cu)
    CU(cudaError_t(deep_launch(H, FIELDS, &k, a, c->sm_count, st)));
    c->launches++;
    return 0;
}

int deep_ready(const physad_ctx* c, const char* what) {
    if (!c->has_weights || c->deep_layers < 1) return fail(PHYSAD_E_NOWEIGHTS, std::string(what) + ": call physad_set_weights_deep first");
    if (c->cfg.In != 4 || c->cfg.Out != 4 || (c->cfg.H != 32 && c->cfg.H != 64 && c->cfg.H != 128))
        return fail(PHYSAD_E_UNSUPPORTED, std::string(what) + ": weights were replaced by a shape the deep kernels are not built for");
    return 0;
}
}  // namespace


// =================================================================================================
extern "C" {

int physad_abi_version(void) { return PHYSAD_ABI_VERSION; }
const char* physad_last_error(void) { return g_err.c_str(); }
const char* physad_error_string(int status) {
    switch (status) {
        case PHYSAD_OK: return "ok";
        case PHYSAD_E_INVALID: return "invalid argument";
        case PHYSAD_E_UNSUPPORTED: return "unsupported shape";
        case PHYSAD_E_NOWEIGHTS: return "no weights set";
        case PHYSAD_E_PEER_TIMEOUT: return "a peer rank never arrived at the in-kernel exchange";
    }
    return status > 0 ? cudaGetErrorString(cudaError_t(status)) : "unknown";
}

int physad_ctx_create(physad_ctx** out, int device) {
    if (!out) return fail(PHYSAD_E_INVALID, "out is null");
    *out = nullptr;
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (ndev == 0) return fail(int(cudaErrorNoDevice), "no CUDA device: this library has no CPU fallback");
    if (device < 0) CU(cudaGetDevice(&device));
    if (device >= ndev) return fail(PHYSAD_E_INVALID, "device index out of range");
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    if (p.major != 10)
        return fail(PHYSAD_E_UNSUPPORTED, std::string("built for sm_100a only; device is sm_") + std::to_string(p.major) +
                                              std::to_string(p.minor));
    DeviceGuard dg(device);
    physad_ctx* c = new physad_ctx();
    c->device = device;
    c->sm_count = p.multiProcessorCount;
    auto init = [c]() -> int {
        CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        CU(cudaMalloc(&c->ticket, sizeof(unsigned int)));
        CU(cudaMemset(c->ticket, 0, sizeof(unsigned int)));
        CU(cudaMalloc(&c->d_acc, 2 * sizeof(double)));
        CU(cudaMallocHost(&c->h_acc, 2 * sizeof(double)));
        CU(cudaHostAlloc(&c->h_res, sizeof(HostResult), cudaHostAllocMapped));
        std::memset(c->h_res, 0, sizeof(HostResult));
        CU(cudaHostGetDevicePointer(reinterpret_cast<void**>(&c->d_res), c->h_res, 0));
        CU(cudaMalloc(&c->d_status, sizeof(unsigned int)));
        CU(cudaMemset(c->d_status, 0, sizeof(unsigned int)));
        return 0;
    };
    if (int rc = init()) {
        const std::string msg = g_err;  // destroy() must not clobber the reason
        physad_ctx_destroy(c);
        return fail(rc, msg);
    }
    *out = c;
    return 0;
}

int physad_ctx_destroy(physad_ctx* c) {
    if (!c) return 0;
    DeviceGuard dg(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    cudaFree(c->dW1); cudaFree(c->db1); cudaFree(c->dW2); cudaFree(c->db2);
    physad_xchg_disconnect(c);
    cudaFree(c->xbuf);
    cudaFree(c->plan.dev);
    cudaFree(c->tab.dev);
    cudaFree(c->d_wh); cudaFree(c->d_bh); cudaFree(c->d_wparts);
    cudaFree(c->partials); cudaFree(c->ticket); cudaFree(c->d_acc); cudaFree(c->scratch);
    cudaFree(c->gws); cudaFree(c->gpart);
    cudaFree(c->dckpt); cudaFree(c->d_dgrad);
    if (c->h_dgrad) cudaFreeHost(c->h_dgrad);
    if (c->h_acc) cudaFreeHost(c->h_acc);
    if (c->h_res) cudaFreeHost(c->h_res);
    cudaFree(c->d_status);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

int physad_ctx_sm_count(const physad_ctx* c) { return c ? c->sm_count : 0; }
uint64_t physad_launch_count(const physad_ctx* c) { return c ? c->launches : 0; }
int physad_set_exact_residuals(physad_ctx* c, int on) {
    if (!c) return -1;
    const int prev = c->exact_residuals;
    c->exact_residuals = on ? 1 : 0;
    return prev;
}
int physad_set_advection(physad_ctx* c, int scheme) {
    if (!c || (scheme != 0 && scheme != 1)) return -1;
    const int prev = c->advection;
    c->advection = scheme;
    return prev;
}
int physad_set_fused_variant(physad_ctx* c, int v) {
    if (!c) return -1;
    const int prev = c->fused_variant;
    c->fused_variant = v;
    return prev;
}

int physad_set_weights(physad_ctx* c, const physad_mlp_config* cfg, const float* W1, const float* b1, const float* W2,
                       const float* b2) {
    if (!c || !cfg || !W1 || !b1 || !W2 || !b2) return fail(PHYSAD_E_INVALID, "set_weights: null argument");
    if (cfg->In <= 0 || cfg->H <= 0 || cfg->Out <= 0) return fail(PHYSAD_E_INVALID, "set_weights: dims must be positive");
    if (cfg->norm != 0 && cfg->norm != 1) return fail(PHYSAD_E_INVALID, "set_weights: norm must be 0 or 1");
    c->cfg = *cfg;
    const size_t n[4] = {size_t(cfg->H) * cfg->In, size_t(cfg->H), size_t(cfg->Out) * cfg->H, size_t(cfg->Out)};
    const float* src[4] = {W1, b1, W2, b2};
    std::vector<float>* host[4] = {&c->W1, &c->b1, &c->W2, &c->b2};
    for (int k = 0; k < 4; ++k) host[k]->assign(src[k], src[k] + n[k]);
    // The grid / fused kernels take the weights through the kernel-parameter block built from this host
    // copy at launch; the device copy is only needed by the explicit-coordinate MLP kernels and is
    // refreshed lazily there.
    c->dev_weights_stale = true;
    c->has_weights = true;
    c->deep_layers = 0;  // a plain set_weights describes a one-hidden-layer network
    return 0;
}


namespace {
// a1[i,h] = relu(b1[h] + sum_k W1[h,k] x[i,k])          (src/mlp_cpu.cpp:18-24)
GemmArgs gemm_hidden(const physad_ctx* c, const float* x, float* act, size_t B) {
    GemmArgs g{};
    const int In = c->cfg.In, H = c->cfg.H;
    g.A = x; g.a_ms = In; g.a_ks = 1; g.B = c->dW1; g.b_ks = 1; g.b_ns = In; g.ones_col = -1; g.init = c->db1;
    g.M = int(B); g.N = H; g.K = In; g.epilogue = GEMM_RELU; g.C = act; g.c_ms = H; g.n_split = H;
    return g;
}
// y[i,o] = b2[o] + sum_h W2[o,h] a1[i,h]   (src/mlp_cpu.cpp:27-34), or gz2 = scale * (y - target) when target != null (:58)
GemmArgs gemm_out(const physad_ctx* c, const float* act, float* out, size_t B, const float* target, float scale) {
    GemmArgs g{};
    const int H = c->cfg.H, Out = c->cfg.Out;
    g.A = act; g.a_ms = H; g.a_ks = 1; g.B = c->dW2; g.b_ks = 1; g.b_ns = H; g.ones_col = -1; g.init = c->db2;
    g.M = int(B); g.N = Out; g.K = H; g.epilogue = target ? GEMM_SCALED_DIFF : GEMM_STORE; g.aux = target; g.scale = scale;
    g.C = out; g.c_ms = Out; g.n_split = Out;
    return g;
}
}  // namespace

// ---- MLP operator -----------------------------------------------------------------------------
int physad_mlp_forward_dev(physad_ctx* c, const float* x, float* y, size_t B, void* stream) {
    if (!c || (B && (!x || !y))) return fail(PHYSAD_E_INVALID, "mlp_forward: null argument");
    if (!c->has_weights) return fail(PHYSAD_E_NOWEIGHTS, "mlp_forward: no weights set");
    if (int rc = need_one_layer(c, "mlp_forward", "physad_mlp_forward_deep_dev")) return rc;
    if (B == 0) return 0;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    const int In = c->cfg.In, H = c->cfg.H, Out = c->cfg.Out;
    const size_t smem4 = size_t(H) * (2 * sizeof(float4) + sizeof(float));
    if (In == 4 && Out == 4 && smem4 <= 200 * 1024 && (uintptr_t(x) % 16 == 0) && (uintptr_t(y) % 16 == 0)) {
        if (smem4 > 48 * 1024)
            CU(cudaFuncSetAttribute(k_mlp_forward_4x4, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem4)));
        k_mlp_forward_4x4<<<unsigned((B + 255) / 256), 256, smem4, st>>>(
            reinterpret_cast<const float4*>(x), c->dW1, c->db1, c->dW2, c->db2, reinterpret_cast<float4*>(y), B, H);
        c->launches++;
    } else {
        if (B > size_t(65535) * 64) return fail(PHYSAD_E_UNSUPPORTED, "mlp_forward: more than 4 194 240 rows per call for generic dims");
        float* act = nullptr;
        CU(cudaMallocAsync(&act, B * size_t(H) * sizeof(float), st));
        CU(cudaError_t(strict_gemm_launch(gemm_hidden(c, x, act, B), st)));
        CU(cudaError_t(strict_gemm_launch(gemm_out(c, act, y, B, nullptr, 0.f), st)));
        c->launches += 2;
        CU(cudaFreeAsync(act, st));
    }
    CU(cudaGetLastError());
    return 0;
}

int physad_mlp_forward_host(physad_ctx* c, const float* x, float* y, size_t B) {
    if (!c || (B && (!x || !y))) return fail(PHYSAD_E_INVALID, "mlp_forward: null argument");
    if (!c->has_weights) return fail(PHYSAD_E_NOWEIGHTS, "mlp_forward: no weights set");
    if (int rc = need_one_layer(c, "mlp_forward", "physad_mlp_forward_deep_dev")) return rc;
    if (B == 0) return 0;
    DeviceGuard dg(c->device);
    Staged a[2] = {{x, nullptr, B * c->cfg.In * sizeof(float)}, {nullptr, y, B * c->cfg.Out * sizeof(float)}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_forward_dev(c, a[0].dev, a[1].dev, B, c->stream)) return rc;
    return stage_out(c, a);
}

int physad_mlp_backward_dev(physad_ctx* c, const float* x, const float* y_target, float* dW1, float* db1, float* dW2,
                            float* db2, size_t B, void* stream) {
    if (!c || !x || !y_target || !dW1 || !db1 || !dW2 || !db2) return fail(PHYSAD_E_INVALID, "mlp_backward: null argument");
    if (!c->has_weights) return fail(PHYSAD_E_NOWEIGHTS, "mlp_backward: no weights set");
    if (int rc = need_one_layer(c, "mlp_backward", "physad_deep_data_loss_grad_dev")) return rc;
    if (B == 0) return fail(PHYSAD_E_INVALID, "mlp_backward: empty batch (the reference divides by B*Out)");
    if (B > size_t(65535) * 64) return fail(PHYSAD_E_UNSUPPORTED, "mlp_backward: more than 4 194 240 rows per call");
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    const int In = c->cfg.In, H = c->cfg.H, Out = c->cfg.Out;
    float *act = nullptr, *gz2 = nullptr, *gz1 = nullptr;
    CU(cudaMallocAsync(&act, B * size_t(H) * sizeof(float), st));
    CU(cudaMallocAsync(&gz1, B * size_t(H) * sizeof(float), st));
    CU(cudaMallocAsync(&gz2, B * size_t(Out) * sizeof(float), st));
    const float scale = 2.f / float(B * size_t(Out));  // src/mlp_cpu.cpp:58
    // five strict contractions (dense_kernels.cuh); every gradient entry is the reference's sequential fp32 sum over the
    // batch, i ascending -- which is also why the batch cannot be split over blocks: partial sums would round differently
    GemmArgs gz1g{}, dw2{}, dw1{};
    // gz1[i,h] = (sum_o gz2[i,o] W2[o,h]) * (a1[i,h] > 0)
    gz1g.A = gz2; gz1g.a_ms = Out; gz1g.a_ks = 1; gz1g.B = c->dW2; gz1g.b_ks = H; gz1g.b_ns = 1; gz1g.ones_col = -1;
    gz1g.M = int(B); gz1g.N = H; gz1g.K = Out; gz1g.epilogue = GEMM_MASK; gz1g.aux = act; gz1g.C = gz1; gz1g.c_ms = H; gz1g.n_split = H;
    // dW2[o,h] = sum_i gz2[i,o] a1[i,h],  db2[o] = sum_i gz2[i,o]  (the extra all-ones column: g * 1 is exact)
    dw2.A = gz2; dw2.a_ms = 1; dw2.a_ks = Out; dw2.B = act; dw2.b_ks = H; dw2.b_ns = 1; dw2.ones_col = H;
    dw2.M = Out; dw2.N = H + 1; dw2.K = int(B); dw2.epilogue = GEMM_STORE; dw2.C = dW2; dw2.c_ms = H; dw2.n_split = H; dw2.C2 = db2;
    // dW1[h,k] = sum_i gz1[i,h] x[i,k],  db1[h] = sum_i gz1[i,h]
    dw1.A = gz1; dw1.a_ms = 1; dw1.a_ks = H; dw1.B = x; dw1.b_ks = In; dw1.b_ns = 1; dw1.ones_col = In;
    dw1.M = H; dw1.N = In + 1; dw1.K = int(B); dw1.epilogue = GEMM_STORE; dw1.C = dW1; dw1.c_ms = In; dw1.n_split = In; dw1.C2 = db1;
    CU(cudaError_t(strict_gemm_launch(gemm_hidden(c, x, act, B), st)));
    CU(cudaError_t(strict_gemm_launch(gemm_out(c, act, gz2, B, y_target, scale), st)));
    CU(cudaError_t(strict_gemm_launch(dw2, st)));
    CU(cudaError_t(strict_gemm_launch(gz1g, st)));
    CU(cudaError_t(strict_gemm_launch(dw1, st)));
    c->launches += 5;
    CU(cudaFreeAsync(act, st));
    CU(cudaFreeAsync(gz1, st));
    CU(cudaFreeAsync(gz2, st));
    return 0;
}

int physad_mlp_backward_host(physad_ctx* c, const float* x, const float* y_target, float* dW1, float* db1, float* dW2,
                             float* db2, size_t B) {
    if (!c || !x || !y_target || !dW1 || !db1 || !dW2 || !db2) return fail(PHYSAD_E_INVALID, "mlp_backward: null argument");
    if (!c->has_weights) return fail(PHYSAD_E_NOWEIGHTS, "mlp_backward: no weights set");
    if (int rc = need_one_layer(c, "mlp_backward", "physad_deep_data_loss_grad_dev")) return rc;
    DeviceGuard dg(c->device);
    const size_t In = c->cfg.In, H = c->cfg.H, Out = c->cfg.Out, f = sizeof(float);
    Staged a[6] = {{x, nullptr, B * In * f}, {y_target, nullptr, B * Out * f}, {nullptr, dW1, H * In * f},
                   {nullptr, db1, H * f}, {nullptr, dW2, Out * H * f}, {nullptr, db2, Out * f}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_backward_dev(c, a[0].dev, a[1].dev, a[2].dev, a[3].dev, a[4].dev, a[5].dev, B, c->stream)) return rc;
    return stage_out(c, a);
}

int physad_mlp_grid_infer_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float* out,
                              void* stream) {
    if (!c || !out) return fail(PHYSAD_E_INVALID, "mlp_grid_infer: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "mlp_grid_infer", "physad_mlp_grid_infer_deep_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    if (uintptr_t(out) % 16) return fail(PHYSAD_E_INVALID, "mlp_grid_infer: out must be 16-byte aligned");
    DeviceGuard dg(c->device);
    const float tcv = time_coord(t, c->cfg.norm);
    const float tc[3] = {tcv, tcv, tcv};
    GridInferArgs a{};
    a.out_aos = reinterpret_cast<float4*>(out);
    return launch_grid<false>(c, g, s, tc, a, cudaStream_t(stream));
}

int physad_mlp_grid_infer_host(physad_ctx* c, const physad_grid* g, float t, float* out) {
    if (!c || !out) return fail(PHYSAD_E_INVALID, "mlp_grid_infer: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    Staged a[1] = {{nullptr, out, size_t(g->nx) * g->ny * g->nz * 4 * sizeof(float)}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_grid_infer_dev(c, g, nullptr, t, a[0].dev, c->stream)) return rc;
    return stage_out(c, a);
}

int physad_mlp_generate_fields_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float dt,
                                   float* s_m, float* s_0, float* s_p, float* u_m, float* u_0, float* u_p, void* stream) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p) return fail(PHYSAD_E_INVALID, "generate_fields: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "generate_fields", "physad_mlp_generate_fields_deep_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    DeviceGuard dg(c->device);
    const float ts[3] = {t - dt, t, t + dt};
    const float tc[3] = {time_coord(ts[0], c->cfg.norm), time_coord(ts[1], c->cfg.norm), time_coord(ts[2], c->cfg.norm)};
    GridInferArgs a{};
    a.sigma[0] = s_m; a.sigma[1] = s_0; a.sigma[2] = s_p;
    a.u[0] = u_m; a.u[1] = u_0; a.u[2] = u_p;
    return launch_grid<true>(c, g, s, tc, a, cudaStream_t(stream));
}

int physad_mlp_generate_fields_host(physad_ctx* c, const physad_grid* g, float t, float dt, float* s_m, float* s_0,
                                    float* s_p, float* u_m, float* u_0, float* u_p) {
    if (!c) return fail(PHYSAD_E_INVALID, "generate_fields: null context");
    if (!s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p) return fail(PHYSAD_E_INVALID, "generate_fields: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    const size_t n = size_t(g->nx) * g->ny * g->nz * sizeof(float);
    Staged a[6] = {{nullptr, s_m, n}, {nullptr, s_0, n}, {nullptr, s_p, n},
                   {nullptr, u_m, 3 * n}, {nullptr, u_0, 3 * n}, {nullptr, u_p, 3 * n}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_generate_fields_dev(c, g, nullptr, t, dt, a[0].dev, a[1].dev, a[2].dev, a[3].dev, a[4].dev, a[5].dev,
                                                c->stream))
        return rc;
    return stage_out(c, a);
}

// ---- deeper MLPs (additive; BASELINE config 5) ------------------------------------------------------
int physad_set_weights_deep(physad_ctx* c, const physad_mlp_config* cfg, int hidden_layers, const float* W1, const float* b1,
                            const float* Wh, const float* bh, const float* W2, const float* b2) {
    if (!c || !cfg) return fail(PHYSAD_E_INVALID, "set_weights_deep: null argument");
    if (cfg->In != 4 || cfg->Out != 4 || (cfg->H != 32 && cfg->H != 64 && cfg->H != 128))
        return fail(PHYSAD_E_UNSUPPORTED, "set_weights_deep: In = Out = 4 and H in {32, 64, 128} are built");
    if (hidden_layers < 1 || hidden_layers > 16) return fail(PHYSAD_E_INVALID, "set_weights_deep: 1 <= hidden_layers <= 16");
    if (hidden_layers > 1 && (!Wh || !bh)) return fail(PHYSAD_E_INVALID, "set_weights_deep: null hidden weights");
    if (int rc = physad_set_weights(c, cfg, W1, b1, W2, b2)) return rc;
    DeviceGuard dg(c->device);
    const size_t H = size_t(cfg->H), nl = size_t(hidden_layers - 1);
    std::vector<float> wt(std::max<size_t>(1, nl * H * H));
    for (size_t l = 0; l < nl; ++l)          // [g][h] row-major -> [h][g] with output pairs stored (g+1, g)
        for (size_t h = 0; h < H; ++h)
            for (size_t g = 0; g < H; g += 2) {
                wt[(l * H + h) * H + g] = Wh[(l * H + g + 1) * H + h];
                wt[(l * H + h) * H + g + 1] = Wh[(l * H + g) * H + h];
            }
    if (int rc = grow(c->d_wh, c->d_wh_cap, wt.size())) return rc;
    if (int rc = grow(c->d_bh, c->d_bh_cap, std::max<size_t>(1, nl * H))) return rc;
    // fast mode (physad_set_deep_mode): every layer as three bf16 terms in the MMA's shared-memory layout
    std::vector<uint8_t> images;
    if (deep_tc_supported(int(H), hidden_layers)) {
        images.resize(nl * deep_tc_layer_bytes(int(H)));
        for (size_t l = 0; l < nl; ++l) deep_tc_pack_layer(int(H), Wh + l * H * H, images.data() + l * deep_tc_layer_bytes(int(H)));
        if (int rc = grow(c->d_wparts, c->d_wparts_cap, images.size())) return rc;
    }
    CU(cudaDeviceSynchronize());   // kernels of ANY stream may still read the previous layers
    if (nl) {
        CU(cudaMemcpy(c->d_wh, wt.data(), nl * H * H * sizeof(float), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->d_bh, bh, nl * H * sizeof(float), cudaMemcpyHostToDevice));
        if (!images.empty()) CU(cudaMemcpy(c->d_wparts, images.data(), images.size(), cudaMemcpyHostToDevice));
    }
    c->deep_tc_ok = !images.empty();
    CU(cudaDeviceSynchronize());   // ... and the copies have landed before a kernel on a non-blocking stream can start
    c->deep_layers = hidden_layers;
    return 0;
}

size_t physad_deep_tc_layer_bytes(int H) { return (H == 32 || H == 64 || H == 128) ? deep_tc_layer_bytes(H) : 0; }

int physad_deep_tc_pack_layer(int H, const float* W, unsigned char* image) {
    if (!W || !image) return fail(PHYSAD_E_INVALID, "deep_tc_pack_layer: null argument");
    if (H != 32 && H != 64 && H != 128) return fail(PHYSAD_E_UNSUPPORTED, "deep_tc_pack_layer: H in {32, 64, 128}");
    deep_tc_pack_layer(H, W, image);
    return 0;
}

int physad_set_deep_mode(physad_ctx* c, int mode) {
    if (!c) return fail(PHYSAD_E_INVALID, "set_deep_mode: null context");
    if (mode != 0 && mode != 1) return fail(PHYSAD_E_INVALID, "set_deep_mode: 0 (strict fp32) or 1 (tensor cores, three-term bf16)");
    c->deep_mode = mode;
    return 0;
}

int physad_mlp_grid_infer_deep_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float* out,
                                   void* stream) {
    if (!c || !out) return fail(PHYSAD_E_INVALID, "mlp_grid_infer_deep: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "mlp_grid_infer_deep")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    if (uintptr_t(out) % 16) return fail(PHYSAD_E_INVALID, "mlp_grid_infer_deep: out must be 16-byte aligned");
    DeviceGuard dg(c->device);
    const float tcv = time_coord(t, c->cfg.norm);
    const float tc[3] = {tcv, tcv, tcv};
    // one hidden layer: the reference-pinned kernel (bit-identical and cheaper); PHYSAD_DEEP_FORCE keeps the deep kernel
    // so that the tests can pin ITS layer-1 / output arithmetic to the reference at L = 1
    if (c->deep_layers == 1 && !getenv("PHYSAD_DEEP_FORCE")) {
        GridInferArgs ga{};
        ga.out_aos = reinterpret_cast<float4*>(out);
        return launch_grid<false>(c, g, s, tc, ga, cudaStream_t(stream));
    }
    DeepArgs a{};
    a.out_aos = reinterpret_cast<float4*>(out);
    switch (c->cfg.H) {
        case 32: return launch_deep<32, false>(c, g, s, tc, a, cudaStream_t(stream));
        case 64: return launch_deep<64, false>(c, g, s, tc, a, cudaStream_t(stream));
        default: return launch_deep<128, false>(c, g, s, tc, a, cudaStream_t(stream));
    }
}

int physad_mlp_generate_fields_deep_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float dt,
                                        float* s_m, float* s_0, float* s_p, float* u_m, float* u_0, float* u_p,
                                        void* stream) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p) return fail(PHYSAD_E_INVALID, "generate_fields_deep: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "generate_fields_deep")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    DeviceGuard dg(c->device);
    const float ts[3] = {t - dt, t, t + dt};
    const float tc[3] = {time_coord(ts[0], c->cfg.norm), time_coord(ts[1], c->cfg.norm), time_coord(ts[2], c->cfg.norm)};
    if (c->deep_layers == 1 && !getenv("PHYSAD_DEEP_FORCE")) {
        GridInferArgs ga{};
        ga.sigma[0] = s_m; ga.sigma[1] = s_0; ga.sigma[2] = s_p;
        ga.u[0] = u_m; ga.u[1] = u_0; ga.u[2] = u_p;
        return launch_grid<true>(c, g, s, tc, ga, cudaStream_t(stream));
    }
    DeepArgs a{};
    a.sigma[0] = s_m; a.sigma[1] = s_0; a.sigma[2] = s_p;
    a.u[0] = u_m; a.u[1] = u_0; a.u[2] = u_p;
    switch (c->cfg.H) {
        case 32: return launch_deep<32, true>(c, g, s, tc, a, cudaStream_t(stream));
        case 64: return launch_deep<64, true>(c, g, s, tc, a, cudaStream_t(stream));
        default: return launch_deep<128, true>(c, g, s, tc, a, cudaStream_t(stream));
    }
}

// one call: deep network -> six fields in context scratch -> residual loss -> the two losses on the host
int physad_deep_loss_host(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, float t, float dt, float* loss_sigma,
                          float* loss_u) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "deep_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "deep_loss")) return rc;
    DeviceGuard dg(c->device);
    const size_t N = size_t(g->nx) * g->ny * g->nz, n = N * sizeof(float);
    Staged f[6] = {{nullptr, nullptr, n}, {nullptr, nullptr, n}, {nullptr, nullptr, n},   // sigma_{-,0,+}, u_{-,0,+}: workspace
                   {nullptr, nullptr, 3 * n}, {nullptr, nullptr, 3 * n}, {nullptr, nullptr, 3 * n}};
    if (int rc = stage_in(c, f)) return rc;
    if (int rc = physad_mlp_generate_fields_deep_dev(c, g, nullptr, t, dt, f[0].dev, f[1].dev, f[2].dev, f[3].dev, f[4].dev, f[5].dev,
                                                     c->stream))
        return rc;
    if (int rc = physad_phys_loss_dev(c, g, f[0].dev, f[1].dev, f[2].dev, f[3].dev, f[4].dev, f[5].dev, c->d_acc, nullptr, nullptr,
                                      nullptr, nullptr, c->stream))
        return rc;
    CU(cudaMemcpyAsync(c->h_acc, c->d_acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    physad_finalize_loss(c->h_acc, w, N, loss_sigma, loss_u);
    return 0;
}

// ---- physics on supplied fields ------------------------------------------------------------------
int physad_phys_residuals_dev(physad_ctx* c, const physad_grid* g, const float* s_m, const float* s_0, const float* s_p,
                              const float* u_m, const float* u_0, const float* u_p, float* Rs, float* Rx, float* Ry,
                              float* Rz, void* stream) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !Rs || !Rx || !Ry || !Rz)
        return fail(PHYSAD_E_INVALID, "phys_residuals: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    return launch_phys<true, false, false>(c, g, phys_args(s_m, s_0, s_p, u_m, u_0, u_p, Rs, Rx, Ry, Rz), cudaStream_t(stream));
}

int physad_phys_loss_dev(physad_ctx* c, const physad_grid* g, const float* s_m, const float* s_0, const float* s_p,
                         const float* u_m, const float* u_0, const float* u_p, double* acc, float* Rs, float* Rx,
                         float* Ry, float* Rz, void* stream) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !acc) return fail(PHYSAD_E_INVALID, "phys_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    PhysArgs a = phys_args(s_m, s_0, s_p, u_m, u_0, u_p, Rs, Rx, Ry, Rz);
    a.acc_out = acc;
    if (Rs || Rx || Ry || Rz) return launch_phys<true, true, false>(c, g, a, cudaStream_t(stream));
    return launch_phys<false, true, false>(c, g, a, cudaStream_t(stream));
}

// ---- reduced-precision field I/O (additive) ----------------------------------------------------------------------
int physad_mlp_generate_fields_lp_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float dt, int dtype,
                                      void* s_m, void* s_0, void* s_p, void* u_m, void* u_0, void* u_p, void* stream) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p) return fail(PHYSAD_E_INVALID, "generate_fields_lp: null argument");
    if (dtype != PHYSAD_F16 && dtype != PHYSAD_BF16) return fail(PHYSAD_E_INVALID, "generate_fields_lp: dtype must be PHYSAD_F16 or PHYSAD_BF16");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "generate_fields_lp", nullptr)) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    DeviceGuard dg(c->device);
    const float ts[3] = {t - dt, t, t + dt};
    const float tc[3] = {time_coord(ts[0], c->cfg.norm), time_coord(ts[1], c->cfg.norm), time_coord(ts[2], c->cfg.norm)};
    GridInferArgs a{};
    a.sigma[0] = static_cast<float*>(s_m); a.sigma[1] = static_cast<float*>(s_0); a.sigma[2] = static_cast<float*>(s_p);
    a.u[0] = static_cast<float*>(u_m); a.u[1] = static_cast<float*>(u_0); a.u[2] = static_cast<float*>(u_p);
    return launch_grid<true>(c, g, s, tc, a, cudaStream_t(stream), dtype);
}

int physad_phys_loss_lp_dev(physad_ctx* c, const physad_grid* g, int dtype, const void* s_m, const void* s_0, const void* s_p,
                            const void* u_m, const void* u_0, const void* u_p, double* acc, float* Rs, float* Rx, float* Ry,
                            float* Rz, void* stream) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !acc) return fail(PHYSAD_E_INVALID, "phys_loss_lp: null argument");
    if (dtype != PHYSAD_F16 && dtype != PHYSAD_BF16) return fail(PHYSAD_E_INVALID, "phys_loss_lp: dtype must be PHYSAD_F16 or PHYSAD_BF16");
    if (int rc = check_grid(g)) return rc;
    if (int rc = check_residual_outputs(Rs, Rx, Ry, Rz, "phys_loss_lp")) return rc;
    DeviceGuard dg(c->device);
    auto f = [](const void* p) { return static_cast<const float*>(p); };   // element type travels in `dtype`
    PhysArgs a = phys_args(f(s_m), f(s_0), f(s_p), f(u_m), f(u_0), f(u_p), Rs, Rx, Ry, Rz);
    a.acc_out = acc;
    if (Rs) return launch_phys<true, true, false>(c, g, a, cudaStream_t(stream), -1, dtype);
    return launch_phys<false, true, false>(c, g, a, cudaStream_t(stream), -1, dtype);
}

int physad_phys_loss_slab_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, const float* s_m,
                              const float* s_0, const float* s_p, const float* u_m, const float* u_0, const float* u_p,
                              const float* halo_lo, const float* halo_hi, double* acc, float* Rs, float* Rx, float* Ry,
                              float* Rz, void* stream) {
    if (!c || !slab || !acc) return fail(PHYSAD_E_INVALID, "phys_loss_slab: null argument");
    if (int rc = check_grid(g)) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    const int nzl = s.z_end - s.z_begin;
    if (nzl > 0 && (!s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !halo_lo || !halo_hi))
        return fail(PHYSAD_E_INVALID, "phys_loss_slab: null field or halo pointer");
    DeviceGuard dg(c->device);
    PhysArgs a = phys_args(s_m, s_0, s_p, u_m, u_0, u_p, Rs, Rx, Ry, Rz);
    a.acc_out = acc;
    a.halo_lo = halo_lo; a.halo_hi = halo_hi;
    if (Rs || Rx || Ry || Rz) return launch_phys<true, true, false>(c, g, a, cudaStream_t(stream), nzl);
    return launch_phys<false, true, false>(c, g, a, cudaStream_t(stream), nzl);
}

int physad_phys_backward_dev(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, const float* Rs,
                             const float* Rx, const float* Ry, const float* Rz, float* gs, float* gx, float* gy,
                             float* gz, void* stream) {
    if (!c || !w || !Rs || !Rx || !Ry || !Rz || !gs || !gx || !gy || !gz)
        return fail(PHYSAD_E_INVALID, "phys_backward: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    ScaleArgs a{};
    float ss, su;
    vjp_scales(g, w, &ss, &su);
    a.R[0] = Rs; a.R[1] = Rx; a.R[2] = Ry; a.R[3] = Rz;
    a.G[0] = gs; a.G[1] = gx; a.G[2] = gy; a.G[3] = gz;
    a.scale[0] = ss; a.scale[1] = a.scale[2] = a.scale[3] = su;
    a.n = size_t(g->nx) * g->ny * g->nz;
    int vec4 = (a.n % 4 == 0);
    for (int k = 0; k < 4; ++k) vec4 = vec4 && (uintptr_t(a.R[k]) % 16 == 0) && (uintptr_t(a.G[k]) % 16 == 0);
    const size_t work = vec4 ? a.n / 4 : a.n;
    const unsigned blocks = unsigned(std::min<size_t>((work + 255) / 256, size_t(c->sm_count) * 16));
    k_scale4<<<std::max(1u, blocks), 256, 0, cudaStream_t(stream)>>>(a, vec4);
    c->launches++;
    CU(cudaGetLastError());
    return 0;
}

int physad_phys_backward_from_fields_dev(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w,
                                         const float* s_m, const float* s_0, const float* s_p, const float* u_m,
                                         const float* u_0, const float* u_p, float* gs, float* gx, float* gy, float* gz,
                                         void* stream) {
    if (!c || !w || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !gs || !gx || !gy || !gz)
        return fail(PHYSAD_E_INVALID, "phys_backward_from_fields: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    PhysArgs a = phys_args(s_m, s_0, s_p, u_m, u_0, u_p, gs, gx, gy, gz);
    vjp_scales(g, w, &a.scale_s, &a.scale_u);
    return launch_phys<true, false, true>(c, g, a, cudaStream_t(stream));
}

// Host-pointer forms: stage 12N floats in, run, stage results out (the reference API's contract,
// include/phys.h:66, minus its per-call allocations: scratch is kept by the context).
int physad_phys_residuals_host(physad_ctx* c, const physad_grid* g, const float* s_m, const float* s_0, const float* s_p,
                               const float* u_m, const float* u_0, const float* u_p, float* Rs, float* Rx, float* Ry,
                               float* Rz, float* kernel_ms) {
    if (!c || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !Rs || !Rx || !Ry || !Rz)
        return fail(PHYSAD_E_INVALID, "phys_residuals: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    const size_t n = size_t(g->nx) * g->ny * g->nz * sizeof(float);
    Staged a[10] = {{s_m, nullptr, n}, {s_0, nullptr, n}, {s_p, nullptr, n}, {u_m, nullptr, 3 * n}, {u_0, nullptr, 3 * n},
                    {u_p, nullptr, 3 * n}, {nullptr, Rs, n}, {nullptr, Rx, n}, {nullptr, Ry, n}, {nullptr, Rz, n}};
    if (int rc = stage_in(c, a)) return rc;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (kernel_ms) {
        CU(cudaEventCreate(&e0));
        CU(cudaEventCreate(&e1));
        CU(cudaEventRecord(e0, c->stream));
    }
    if (int rc = physad_phys_residuals_dev(c, g, a[0].dev, a[1].dev, a[2].dev, a[3].dev, a[4].dev, a[5].dev, a[6].dev, a[7].dev,
                                           a[8].dev, a[9].dev, c->stream))
        return rc;
    if (kernel_ms) CU(cudaEventRecord(e1, c->stream));
    if (int rc = stage_out(c, a)) return rc;
    if (kernel_ms) {
        CU(cudaEventElapsedTime(kernel_ms, e0, e1));
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    }
    return 0;
}

int physad_phys_loss_host(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, const float* s_m,
                          const float* s_0, const float* s_p, const float* u_m, const float* u_0, const float* u_p,
                          float* loss_sigma, float* loss_u, float* Rs, float* Rx, float* Ry, float* Rz) {
    if (!c || !w || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p) return fail(PHYSAD_E_INVALID, "phys_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    const size_t N = size_t(g->nx) * g->ny * g->nz, n = N * sizeof(float);
    Staged a[10] = {{s_m, nullptr, n}, {s_0, nullptr, n}, {s_p, nullptr, n}, {u_m, nullptr, 3 * n}, {u_0, nullptr, 3 * n},
                    {u_p, nullptr, 3 * n}, {nullptr, Rs, n}, {nullptr, Rx, n}, {nullptr, Ry, n}, {nullptr, Rz, n}};
    if (int rc = stage_in(c, a)) return rc;
    float* dev_r[4];
    for (int k = 0; k < 4; ++k) dev_r[k] = a[6 + k].down ? a[6 + k].dev : nullptr;
    if (int rc = physad_phys_loss_dev(c, g, a[0].dev, a[1].dev, a[2].dev, a[3].dev, a[4].dev, a[5].dev, c->d_acc, dev_r[0],
                                      dev_r[1], dev_r[2], dev_r[3], c->stream))
        return rc;
    CU(cudaMemcpyAsync(c->h_acc, c->d_acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (int rc = stage_out(c, a)) return rc;
    physad_finalize_loss(c->h_acc, w, N, loss_sigma, loss_u);
    return 0;
}

int physad_phys_backward_host(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, const float* Rs,
                              const float* Rx, const float* Ry, const float* Rz, float* gs, float* gx, float* gy,
                              float* gz) {
    if (!c || !w || !Rs || !Rx || !Ry || !Rz || !gs || !gx || !gy || !gz)
        return fail(PHYSAD_E_INVALID, "phys_backward: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    const size_t n = size_t(g->nx) * g->ny * g->nz * sizeof(float);
    Staged a[8] = {{Rs, nullptr, n}, {Rx, nullptr, n}, {Ry, nullptr, n}, {Rz, nullptr, n},
                   {nullptr, gs, n}, {nullptr, gx, n}, {nullptr, gy, n}, {nullptr, gz, n}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_phys_backward_dev(c, g, w, a[0].dev, a[1].dev, a[2].dev, a[3].dev, a[4].dev, a[5].dev, a[6].dev, a[7].dev,
                                          c->stream))
        return rc;
    return stage_out(c, a);
}

int physad_phys_backward_from_fields_host(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w,
                                          const float* s_m, const float* s_0, const float* s_p, const float* u_m,
                                          const float* u_0, const float* u_p, float* gs, float* gx, float* gy, float* gz) {
    if (!c || !w || !s_m || !s_0 || !s_p || !u_m || !u_0 || !u_p || !gs || !gx || !gy || !gz)
        return fail(PHYSAD_E_INVALID, "phys_backward_from_fields: null argument");
    if (int rc = check_grid(g)) return rc;
    DeviceGuard dg(c->device);
    const size_t n = size_t(g->nx) * g->ny * g->nz * sizeof(float);
    Staged a[10] = {{s_m, nullptr, n}, {s_0, nullptr, n}, {s_p, nullptr, n}, {u_m, nullptr, 3 * n}, {u_0, nullptr, 3 * n},
                    {u_p, nullptr, 3 * n}, {nullptr, gs, n}, {nullptr, gx, n}, {nullptr, gy, n}, {nullptr, gz, n}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_phys_backward_from_fields_dev(c, g, w, a[0].dev, a[1].dev, a[2].dev, a[3].dev, a[4].dev, a[5].dev,
                                                      a[6].dev, a[7].dev, a[8].dev, a[9].dev, c->stream))
        return rc;
    return stage_out(c, a);
}

// ---- the metric path ---------------------------------------------------------------------------------
int physad_fused_loss_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float dt, double* acc,
                          float* Rs, float* Rx, float* Ry, float* Rz, void* stream) {
    if (!c || !acc) return fail(PHYSAD_E_INVALID, "fused_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "fused_loss", "physad_deep_loss_host or physad_deep_loss_grad_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    if (int rc = check_residual_outputs(Rs, Rx, Ry, Rz, "fused_loss")) return rc;
    DeviceGuard dg(c->device);
    float* R[4] = {Rs, Rx, Ry, Rz};
    return launch_fused(c, g, s, t, dt, acc, R, cudaStream_t(stream));
}

int physad_fused_loss_allreduce_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, float dt,
                                    double* acc, float* Rs, float* Rx, float* Ry, float* Rz, void* stream) {
    if (!c || !acc) return fail(PHYSAD_E_INVALID, "fused_loss_allreduce: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "fused_loss_allreduce", "physad_deep_loss_grad_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    if (int rc = check_residual_outputs(Rs, Rx, Ry, Rz, "fused_loss_allreduce")) return rc;
    DeviceGuard dg(c->device);
    float* R[4] = {Rs, Rx, Ry, Rz};
    return launch_fused(c, g, s, t, dt, acc, R, cudaStream_t(stream), true);
}

// ---- analytic (tangent) loss: derivatives propagated through the MLP in forward mode (additive, NOT the parity path) ----
}  // extern "C"  (templates below)
namespace {
template <int H>
void fill_tangent(const physad_ctx* c, float tcoord, TangentConst<H>& k) {
    const int h_rt = c->cfg.H;
    for (int h = 0; h < H; ++h) {
        const bool on = h < h_rt;
        const float w1[4] = {on ? c->W1[size_t(h) * 4] : 0.f, on ? c->W1[size_t(h) * 4 + 1] : 0.f, on ? c->W1[size_t(h) * 4 + 2] : 0.f,
                             on ? c->W1[size_t(h) * 4 + 3] : 0.f};
        volatile float pt = w1[3] * tcoord;   // separately rounded product, as MlpConst::pt0
        k.w1[h] = make_float4(w1[0], w1[1], w1[2], float(pt));
        k.b1[h] = on ? c->b1[h] : 0.f;        // padded units: z = 0, mask 0, contribute nothing
        float w2[4];
        for (int o = 0; o < 4; ++o) w2[o] = on ? c->W2[size_t(o) * h_rt + h] : 0.f;
        k.w2[h] = make_float4(w2[0], w2[1], w2[2], w2[3]);
        for (int o = 0; o < 4; ++o) k.p[h][o] = make_float4(w2[o] * w1[0], w2[o] * w1[1], w2[o] * w1[2], w2[o] * w1[3]);
    }
    k.b2 = make_float4(c->b2[0], c->b2[1], c->b2[2], c->b2[3]);
}

template <int H>
int launch_tangent_t(physad_ctx* c, const TangentArgs& a, float tcoord, int blocks, cudaStream_t st) {
    TangentConst<H> k;
    fill_tangent<H>(c, tcoord, k);
    CU(cudaError_t(tangent_launch(H, &k, a, blocks, st)));
    c->launches++;
    return 0;
}
}  // namespace
extern "C" {

int physad_tangent_loss_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, double* acc, float* Rs,
                            float* Rx, float* Ry, float* Rz, void* stream) {
    if (!c || !acc) return fail(PHYSAD_E_INVALID, "tangent_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "tangent_loss", "physad_deep_tangent_loss_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    if (int rc = check_residual_outputs(Rs, Rx, Ry, Rz, "tangent_loss")) return rc;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (s.z_end == s.z_begin) return zero_result(acc, 2, nullptr, 0, st);
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    TangentArgs a{};
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz; a.z_begin = s.z_begin; a.z_end = s.z_end;
    a.cxs = c->tab.dev; a.cys = a.cxs + g->nx; a.czs = a.cys + g->ny;
    float s3[3];
    input_scales(g, c->cfg.norm, s3);
    a.sx = s3[0]; a.sy = s3[1]; a.sz = s3[2];
    const size_t n = size_t(s.z_end - s.z_begin) * g->ny * g->nx;
    const int blocks = int(std::max<size_t>(1, std::min<size_t>(size_t(c->sm_count) * 2, (n + 2 * TANGENT_THREADS - 1) / (2 * TANGENT_THREADS))));
    if (int rc = ensure_partials(c, size_t(blocks))) return rc;
    a.partials = c->partials; a.ticket = c->ticket; a.acc_out = acc;
    a.R[0] = Rs; a.R[1] = Rx; a.R[2] = Ry; a.R[3] = Rz;
    const float tc = time_coord(t, c->cfg.norm);
    switch (template_h(c->cfg.H)) {
        case 32: return launch_tangent_t<32>(c, a, tc, blocks, st);
        case 64: return launch_tangent_t<64>(c, a, tc, blocks, st);
        case 128: return launch_tangent_t<128>(c, a, tc, blocks, st);
    }
    return fail(PHYSAD_E_UNSUPPORTED, "H > 128 not built");
}

int physad_tangent_loss_host(physad_ctx* c, const physad_grid* g, const physad_mlp_config* cfg, const float* W1, const float* b1,
                             const float* W2, const float* b2, const physad_phys_weights* w, float t, float* loss_sigma,
                             float* loss_u) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "tangent_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    if (cfg) {
        if (int rc = physad_set_weights(c, cfg, W1, b1, W2, b2)) return rc;
    }
    DeviceGuard dg(c->device);
    if (int rc = physad_tangent_loss_dev(c, g, nullptr, t, c->d_acc, nullptr, nullptr, nullptr, nullptr, c->stream)) return rc;
    CU(cudaMemcpyAsync(c->h_acc, c->d_acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    physad_finalize_loss(c->h_acc, w, size_t(g->nx) * g->ny * g->nz, loss_sigma, loss_u);
    return 0;
}

// ---- closed loop: loss and its gradient with respect to the MLP weights (additive, grad_kernels.cuh) ----

namespace {
// The closed loops' workspace for NL points in gws: the six fields sigma_{-,0,+} (NL each) and u_{-,0,+} (3 NL each), the
// four residuals R[k] = R + k NL, and the time-t output adjoint (4 NL)
struct LoopWorkspace {
    float *s_m, *s_0, *s_p, *u_m, *u_0, *u_p, *R;
    float4* adj;
};

int loop_workspace(physad_ctx* c, size_t NL, LoopWorkspace& w) {
    if (int rc = grow(c->gws, c->gws_cap, 20 * NL)) return rc;
    float* f = c->gws;
    w = {f, f + NL, f + 2 * NL, f + 3 * NL, f + 6 * NL, f + 9 * NL, f + 12 * NL, reinterpret_cast<float4*>(f + 16 * NL)};
    return 0;
}

// The lengths of the gradient's six arrays in physad_set_weights_deep's order dW1, db1, dWh, dbh, dW2, db2 for the context's
// network; returns their sum P.  With one hidden layer dWh and dbh are empty: the layout dW1 | db1 | dW2 | db2 of any width.
size_t grad_parts(const physad_ctx* c, size_t len[6]) {
    const size_t nl = size_t(std::max(1, c->deep_layers) - 1), H = size_t(c->cfg.H);
    const size_t l[6] = {4 * H, H, nl * H * H, nl * H, 4 * H, 4};
    std::copy(l, l + 6, len);
    return 9 * H + 4 + nl * (H * H + H);
}

// The host forms of the gradients: the context's device result buffer d_dgrad [acc | grad] (at most 2 sums + P) and its
// pinned host copy h_dgrad ...
int ensure_host_grad(physad_ctx* c) {
    size_t len[6];
    const size_t n = grad_parts(c, len) + 2;
    if (int rc = grow(c->d_dgrad, c->d_dgrad_cap, n)) return rc;
    return grow(c->h_dgrad, c->h_dgrad_cap, n, true);
}

// ... and the way back: one copy of [acc (nacc sums) | grad (P)] into h_dgrad, one stream synchronisation, then the loss
// -- physad_finalize_loss of the two physics sums over n points (nacc = 2), the fit loss acc / n (nacc = 1), none for the
// VJPs (nacc = 0) -- and the gradient split into physad_set_weights_deep's six arrays dW1, db1, dWh, dbh, dW2, db2 (a null
// array is skipped; at one hidden layer dWh and dbh are empty)
int grad_to_host(physad_ctx* c, int nacc, size_t n, const physad_phys_weights* w, float* loss_a, float* loss_b,
                 const std::array<float*, 6>& out) {
    size_t len[6];
    const size_t P = grad_parts(c, len);
    CU(cudaMemcpyAsync(c->h_dgrad, c->d_dgrad, (nacc + P) * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (nacc == 2) physad_finalize_loss(c->h_dgrad, w, n, loss_a, loss_b);
    if (nacc == 1 && loss_a) *loss_a = float(c->h_dgrad[0] / double(n));
    const double* gd = c->h_dgrad + nacc;
    for (int k = 0; k < 6; ++k) {
        if (out[k]) for (size_t i = 0; i < len[k]; ++i) out[k][i] = float(gd[i]);
        gd += len[k];
    }
    return 0;
}

// the parts of GradArgs that do not depend on where the arrays live
int grad_args_common(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, float t, float dt, GradArgs& a,
                     cudaStream_t st) {
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz;
    a.periodic = g->periodic != 0;
    a.cxs = c->tab.dev; a.cys = a.cxs + g->nx; a.czs = a.cys + g->ny;
    vjp_scales(g, w, &a.scale_s, &a.scale_u);
    // the residual's time derivative uses GridSpec::dt (src/phys_cpu.cpp:38), like every forward path here; the
    // call's `dt` only places the three slices (src/mlp_grid.cpp:87-89) -- the two are independent in the reference API
    a.inv2dt = inv2(g->dt); a.inv2hx = inv2(g->hx); a.inv2hy = inv2(g->hy); a.inv2hz = inv2(g->hz);
    const float ts[3] = {t - dt, t, t + dt};
    for (int k = 0; k < 3; ++k) a.tc[k] = time_coord(ts[k], c->cfg.norm);
    a.W1 = c->dW1; a.b1 = c->db1; a.W2 = c->dW2;
    a.H = c->cfg.H;
    a.ticket = c->ticket;
    return 0;
}
}  // namespace

int physad_fused_loss_grad_dev(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, float t, float dt,
                               double* acc, double* grad, void* stream) {
    if (!c || !w || !acc || !grad) return fail(PHYSAD_E_INVALID, "fused_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "fused_loss_grad", "physad_deep_loss_grad_dev")) return rc;
    if (c->advection != 0) return fail(PHYSAD_E_UNSUPPORTED, "fused_loss_grad: the stencil adjoint is that of the central scheme");
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    const size_t N = size_t(g->nx) * g->ny * g->nz;
    LoopWorkspace f;
    if (int rc = loop_workspace(c, N, f)) return rc;
    // forward, stage-wise on the device: fields of the three slices, then residuals + the two sums
    float* R = f.R;
    if (int rc = physad_mlp_generate_fields_dev(c, g, nullptr, t, dt, f.s_m, f.s_0, f.s_p, f.u_m, f.u_0, f.u_p, stream)) return rc;
    if (int rc = physad_phys_loss_dev(c, g, f.s_m, f.s_0, f.s_p, f.u_m, f.u_0, f.u_p, acc, R, R + N, R + 2 * N, R + 3 * N, stream))
        return rc;
    // backward
    GradArgs a{};
    if (int rc = grad_args_common(c, g, w, t, dt, a, st)) return rc;
    a.z_begin = 0; a.z_end = g->nz; a.z_origin = 0;
    a.wrap_z = a.periodic;
    a.cstride = N;
    a.s0 = f.s_0; a.u0 = f.u_0;
    for (int k = 0; k < 4; ++k) a.R[k] = R + k * N;
    a.grad = grad;
    return launch_grad(c, template_h(c->cfg.H), a, f.adj, (N + GRAD_THREADS - 1) / GRAD_THREADS, st);
}

int physad_fused_loss_grad_slab_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab,
                                    const physad_phys_weights* w, float t, float dt, double* acc, double* grad, void* stream) {
    if (!c || !w || !acc || !grad || !slab) return fail(PHYSAD_E_INVALID, "fused_loss_grad_slab: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "fused_loss_grad_slab", "physad_deep_loss_grad_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    if (s.z_begin == 0 && s.z_end == g->nz) return physad_fused_loss_grad_dev(c, g, w, t, dt, acc, grad, stream);
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    const int H = c->cfg.H;
    if (c->advection != 0) return fail(PHYSAD_E_UNSUPPORTED, "fused_loss_grad_slab: the stencil adjoint is that of the central scheme");
    if (s.z_begin == s.z_end) return zero_result(acc, 2, grad, size_t(9 * H + 4), st);
    // The gradient of the slab's points needs the residuals one plane beyond the slab, hence the fields two planes
    // beyond it: a window of VIRTUAL planes [zlo, zhi) (wrapped on a periodic grid, cut at the faces otherwise) is
    // recomputed locally -- no halo exchange, like the forward path (SURVEY.md 8e).
    const bool per = g->periodic != 0;
    const int zlo = per ? s.z_begin - 2 : std::max(0, s.z_begin - 2);
    const int zhi = per ? s.z_end + 2 : std::min(g->nz, s.z_end + 2);
    const int npl = zhi - zlo;
    const size_t pln = size_t(g->nx) * g->ny, NL = pln * npl;
    if (NL >= (size_t(1) << 31)) return fail(PHYSAD_E_UNSUPPORTED, "fused_loss_grad_slab: window of 2^31 points or more");
    LoopWorkspace f;
    if (int rc = loop_workspace(c, NL, f)) return rc;
    float* R = f.R;
    const float ts[3] = {t - dt, t, t + dt};
    const float tc[3] = {time_coord(ts[0], c->cfg.norm), time_coord(ts[1], c->cfg.norm), time_coord(ts[2], c->cfg.norm)};
    // fields: one launch per run of consecutive global planes inside the window
    for (int zv = zlo; zv < zhi;) {
        const int ga = ((zv % g->nz) + g->nz) % g->nz;
        const int run = std::min(zhi - zv, g->nz - ga);
        const size_t off = size_t(zv - zlo) * pln;
        GridInferArgs ga_args{};
        ga_args.sigma[0] = f.s_m + off; ga_args.sigma[1] = f.s_0 + off; ga_args.sigma[2] = f.s_p + off;
        ga_args.u[0] = f.u_m + off; ga_args.u[1] = f.u_0 + off; ga_args.u[2] = f.u_p + off;
        ga_args.cstride = NL;
        if (int rc = launch_grid<true>(c, g, physad_slab{ga, ga + run}, tc, ga_args, st)) return rc;
        zv += run;
    }
    // residuals of every plane of the window with the z neighbours clamped at its ends: exact wherever both z
    // neighbours are inside the window (or the end is a face of a non-periodic grid); the other planes are not used
    PhysArgs pa = phys_args(f.s_m, f.s_0, f.s_p, f.u_m, f.u_0, f.u_p, R, R + NL, R + 2 * NL, R + 3 * NL);
    pa.clamp_z = 1;
    if (int rc = launch_phys<true, false, false>(c, g, pa, st, npl)) return rc;
    GradArgs a{};
    if (int rc = grad_args_common(c, g, w, t, dt, a, st)) return rc;
    a.z_begin = s.z_begin; a.z_end = s.z_end; a.z_origin = zlo;
    a.wrap_z = 0;
    a.cstride = NL;
    a.s0 = f.s_0; a.u0 = f.u_0;
    for (int k = 0; k < 4; ++k) a.R[k] = R + k * NL;
    a.grad = grad;
    a.acc_out = acc;
    return launch_grad(c, template_h(H), a, f.adj, (pln * size_t(s.z_end - s.z_begin) + GRAD_THREADS - 1) / GRAD_THREADS, st);
}

int physad_fused_loss_grad_host(physad_ctx* c, const physad_grid* g, const physad_mlp_config* cfg, const float* W1,
                                const float* b1, const float* W2, const float* b2, const physad_phys_weights* w, float t,
                                float dt, float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dW2, float* db2) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "fused_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (cfg) {
        if (int rc = physad_set_weights(c, cfg, W1, b1, W2, b2)) return rc;
    }
    if (int rc = need_4x4(c, "fused_loss_grad", "physad_deep_loss_grad_dev")) return rc;
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    if (int rc = physad_fused_loss_grad_dev(c, g, w, t, dt, c->d_dgrad, c->d_dgrad + 2, c->stream)) return rc;
    return grad_to_host(c, 2, size_t(g->nx) * g->ny * g->nz, w, loss_sigma, loss_u, {dW1, db1, nullptr, nullptr, dW2, db2});
}

// ---- closed loop of the analytic loss: its gradient with respect to the MLP weights (tangent_grad_kernels.cuh) ----
}  // extern "C"  (templates below)
namespace {
template <int H>
int launch_tangent_grad_t(physad_ctx* c, const TangentGradArgs& a, float tcoord, size_t chunks, cudaStream_t st) {
    int& bps = c->tgrad_blocks_per_sm[H == 32 ? 0 : (H == 64 ? 1 : 2)];
    if (!bps) {
        CU(cudaError_t(tangent_grad_blocks_per_sm(H, &bps)));
        if (bps < 1) return fail(PHYSAD_E_UNSUPPORTED, "tangent_loss_grad: kernel does not fit an SM");
    }
    const size_t blocks = std::max<size_t>(1, std::min<size_t>(chunks, size_t(c->sm_count) * bps));
    if (int rc = ensure_grad_partials(c, blocks * (TGRAD_NACC * H + 6))) return rc;
    TangentGradArgs k = a;
    k.partials = c->gpart;
    TangentConst<H> w;
    fill_tangent<H>(c, tcoord, w);
    CU(cudaError_t(tangent_grad_launch(H, &w, k, unsigned(blocks), st)));
    c->launches++;
    return 0;
}
}  // namespace
extern "C" {

int physad_tangent_loss_grad_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, const physad_phys_weights* w,
                                 float t, double* acc, double* grad, void* stream) {
    if (!c || !w || !acc || !grad) return fail(PHYSAD_E_INVALID, "tangent_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = need_4x4(c, "tangent_loss_grad", "physad_deep_tangent_loss_grad_dev")) return rc;
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    const int H = c->cfg.H;
    if (s.z_end == s.z_begin) return zero_result(acc, 2, grad, size_t(9 * H + 4), st);
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    TangentGradArgs a{};
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz; a.z_begin = s.z_begin; a.z_end = s.z_end;
    a.cxs = c->tab.dev; a.cys = a.cxs + g->nx; a.czs = a.cys + g->ny;
    float s3[3];
    input_scales(g, c->cfg.norm, s3);
    a.sx = s3[0]; a.sy = s3[1]; a.sz = s3[2];
    vjp_scales(g, w, &a.scale_s, &a.scale_u);   // 2 w / float(N) of the whole grid: slab results add up to the grid's
    a.ct = time_coord(t, c->cfg.norm);
    a.W1 = c->dW1; a.W2 = c->dW2;
    a.H = H;
    a.ticket = c->ticket;
    a.acc = acc; a.grad = grad;
    const size_t chunks = (size_t(s.z_end - s.z_begin) * g->ny * g->nx + TGRAD_THREADS - 1) / TGRAD_THREADS;
    switch (template_h(H)) {
        case 32: return launch_tangent_grad_t<32>(c, a, a.ct, chunks, st);
        case 64: return launch_tangent_grad_t<64>(c, a, a.ct, chunks, st);
        case 128: return launch_tangent_grad_t<128>(c, a, a.ct, chunks, st);
    }
    return fail(PHYSAD_E_UNSUPPORTED, "H > 128 not built");
}

int physad_tangent_loss_grad_host(physad_ctx* c, const physad_grid* g, const physad_mlp_config* cfg, const float* W1,
                                  const float* b1, const float* W2, const float* b2, const physad_phys_weights* w, float t,
                                  float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dW2, float* db2) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "tangent_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (cfg) {
        if (int rc = physad_set_weights(c, cfg, W1, b1, W2, b2)) return rc;
    }
    if (int rc = need_4x4(c, "tangent_loss_grad", "physad_deep_tangent_loss_grad_dev")) return rc;
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    if (int rc = physad_tangent_loss_grad_dev(c, g, nullptr, w, t, c->d_dgrad, c->d_dgrad + 2, c->stream)) return rc;
    return grad_to_host(c, 2, size_t(g->nx) * g->ny * g->nz, w, loss_sigma, loss_u, {dW1, db1, nullptr, nullptr, dW2, db2});
}

// ---- closed loop of deeper networks (deep_grad_kernels.cuh) ----------------------------------------------------------
size_t physad_deep_grad_len(int H, int hidden_layers) { return deep_grad_len(H, hidden_layers); }

int physad_deep_loss_grad_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, const physad_phys_weights* w,
                              float t, float dt, double* acc, double* grad, void* stream) {
    if (!c || !w || !acc || !grad) return fail(PHYSAD_E_INVALID, "deep_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "deep_loss_grad")) return rc;
    if (c->deep_mode != 0)
        return fail(PHYSAD_E_UNSUPPORTED, "deep_loss_grad: the gradient is of the strict fp32 network (set_deep_mode(0))");
    if (c->advection != 0) return fail(PHYSAD_E_UNSUPPORTED, "deep_loss_grad: the stencil adjoint is that of the central scheme");
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    const bool whole = s.z_begin == 0 && s.z_end == g->nz;
    // one hidden layer: the one-hidden-layer closed loop, whose gradient layout is the same
    if (c->deep_layers == 1)
        return whole ? physad_fused_loss_grad_dev(c, g, w, t, dt, acc, grad, stream)
                     : physad_fused_loss_grad_slab_dev(c, g, &s, w, t, dt, acc, grad, stream);
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    const int H = c->cfg.H, L = c->deep_layers;
    const size_t P = deep_grad_len(H, L);
    if (s.z_begin == s.z_end) return zero_result(acc, 2, grad, P, st);
    // window of VIRTUAL planes [zlo, zhi) whose fields the slab's gradient needs (as physad_fused_loss_grad_slab_dev)
    const bool per = g->periodic != 0;
    const int zlo = whole ? 0 : (per ? s.z_begin - 2 : std::max(0, s.z_begin - 2));
    const int zhi = whole ? g->nz : (per ? s.z_end + 2 : std::min(g->nz, s.z_end + 2));
    const int npl = zhi - zlo;
    const size_t pln = size_t(g->nx) * g->ny, NL = pln * npl;
    if (NL >= (size_t(1) << 31)) return fail(PHYSAD_E_UNSUPPORTED, "deep_loss_grad: window of 2^31 points or more");
    LoopWorkspace f;
    if (int rc = loop_workspace(c, NL, f)) return rc;
    float* R = f.R;
    if (whole) {
        // the arithmetic of physad_deep_loss_host: same fields, same residual kernel, same sums
        if (int rc = physad_mlp_generate_fields_deep_dev(c, g, nullptr, t, dt, f.s_m, f.s_0, f.s_p, f.u_m, f.u_0, f.u_p, stream))
            return rc;
        if (int rc = physad_phys_loss_dev(c, g, f.s_m, f.s_0, f.s_p, f.u_m, f.u_0, f.u_p, acc, R, R + NL, R + 2 * NL, R + 3 * NL,
                                          stream))
            return rc;
    } else {
        // fields: the deep kernel writes u with the channel stride of its own launch, so each run of consecutive global
        // planes goes to a contiguous scratch buffer and its 12 channel blocks are copied into the window arrays
        int max_run = 0;
        for (int zv = zlo; zv < zhi;) {
            const int ga = ((zv % g->nz) + g->nz) % g->nz, run = std::min(zhi - zv, g->nz - ga);
            max_run = std::max(max_run, run);
            zv += run;
        }
        if (int rc = ensure_scratch(c, 12 * pln * size_t(max_run) * sizeof(float))) return rc;
        float* sc = reinterpret_cast<float*>(c->scratch);
        for (int zv = zlo; zv < zhi;) {
            const int ga = ((zv % g->nz) + g->nz) % g->nz, run = std::min(zhi - zv, g->nz - ga);
            const size_t nr = pln * size_t(run), off = size_t(zv - zlo) * pln;
            const physad_slab rs{ga, ga + run};
            if (int rc = physad_mlp_generate_fields_deep_dev(c, g, &rs, t, dt, sc, sc + nr, sc + 2 * nr, sc + 3 * nr, sc + 6 * nr,
                                                             sc + 9 * nr, stream))
                return rc;
            float* dst[12] = {f.s_m + off, f.s_0 + off, f.s_p + off};
            for (int k = 0; k < 3; ++k)
                for (int ch = 0; ch < 3; ++ch) dst[3 + 3 * k + ch] = (k == 0 ? f.u_m : (k == 1 ? f.u_0 : f.u_p)) + ch * NL + off;
            for (int b = 0; b < 12; ++b)
                CU(cudaMemcpyAsync(dst[b], sc + size_t(b) * nr, nr * sizeof(float), cudaMemcpyDeviceToDevice, st));
            zv += run;
        }
        // residuals of every window plane with the z neighbours clamped at its ends (exact on the planes the slab uses)
        PhysArgs pa = phys_args(f.s_m, f.s_0, f.s_p, f.u_m, f.u_0, f.u_p, R, R + NL, R + 2 * NL, R + 3 * NL);
        pa.clamp_z = 1;
        if (int rc = launch_phys<true, false, false>(c, g, pa, st, npl)) return rc;
    }
    // time-t output adjoint A_t of the slab's points
    GradArgs ga{};
    if (int rc = grad_args_common(c, g, w, t, dt, ga, st)) return rc;
    ga.z_begin = s.z_begin; ga.z_end = s.z_end; ga.z_origin = zlo;
    ga.wrap_z = whole ? ga.periodic : 0;
    ga.cstride = NL;
    ga.s0 = f.s_0; ga.u0 = f.u_0;
    for (int k = 0; k < 4; ++k) ga.R[k] = R + k * NL;
    CU(cudaError_t(adjoint_launch(ga, f.adj, st)));
    c->launches++;
    // back-propagation through every layer, then the block-order reduction
    const long long npts = (long long)pln * (s.z_end - s.z_begin);
    const int blocks = deep_grad_blocks(H, npts, c->sm_count);
    if (int rc = grow(c->dckpt, c->dckpt_cap, size_t(blocks) * deep_grad_ckpt_floats(H, L))) return rc;
    if (int rc = ensure_grad_partials(c, size_t(blocks) * (P + 2))) return rc;
    DeepGradArgs a{};
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz;
    a.z_begin = s.z_begin; a.z_end = s.z_end; a.z_origin = zlo;
    a.hidden_layers = L;
    a.cxs = ga.cxs; a.cys = ga.cys; a.czs = ga.czs;
    a.W1 = c->dW1; a.b1 = c->db1; a.W2 = c->dW2;
    for (int k = 0; k < 3; ++k) a.tc[k] = ga.tc[k];
    a.wh = c->d_wh; a.bh = c->d_bh;
    for (int k = 0; k < 4; ++k) a.R[k] = ga.R[k];
    a.adj = f.adj;
    a.scale_s = ga.scale_s; a.scale_u = ga.scale_u; a.inv2dt = ga.inv2dt;
    a.ckpt = c->dckpt;
    a.partials = c->gpart;
    CU(cudaError_t(deep_grad_launch(H, a, blocks, grad, whole ? nullptr : acc, st)));
    c->launches += 2;
    return 0;
}

int physad_deep_loss_grad_host(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, float t, float dt,
                               float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dWh, float* dbh, float* dW2,
                               float* db2) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "deep_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "deep_loss_grad")) return rc;
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    if (int rc = physad_deep_loss_grad_dev(c, g, nullptr, w, t, dt, c->d_dgrad, c->d_dgrad + 2, c->stream)) return rc;
    return grad_to_host(c, 2, size_t(g->nx) * g->ny * g->nz, w, loss_sigma, loss_u, {dW1, db1, dWh, dbh, dW2, db2});
}

// ---- analytic loss of deeper networks and its closed loop (deep_tangent_kernels.cuh) ---------------------------------
}  // extern "C"  (helpers below)
namespace {
// checks and arguments shared by the loss and the loss + gradient call; *npts = 0 for an empty slab
int deep_tangent_args(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, const char* what,
                      DeepTangentArgs& a, long long* npts, cudaStream_t st) {
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, what)) return rc;
    if (c->deep_mode != 0)
        return fail(PHYSAD_E_UNSUPPORTED, std::string(what) + ": the analytic deep loss is that of the strict fp32 network (set_deep_mode(0))");
    physad_slab s;
    if (int rc = check_slab(g, slab, &s)) return rc;
    const size_t n = size_t(s.z_end - s.z_begin) * g->ny * g->nx;   // < 2^31: check_grid bounds the whole grid
    *npts = (long long)n;
    if (n == 0) return 0;
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    if (int rc = ensure_coord_tables(c, g, st)) return rc;
    a.nx = g->nx; a.ny = g->ny; a.nz = g->nz; a.z_begin = s.z_begin; a.z_end = s.z_end;
    a.hidden_layers = c->deep_layers;
    a.cxs = c->tab.dev; a.cys = a.cxs + g->nx; a.czs = a.cys + g->ny;
    a.W1 = c->dW1; a.b1 = c->db1; a.W2 = c->dW2; a.b2 = c->db2;
    a.wh = c->d_wh; a.bh = c->d_bh;
    a.tc = time_coord(t, c->cfg.norm);
    float s3[3];
    input_scales(g, c->cfg.norm, s3);
    a.sx = s3[0]; a.sy = s3[1]; a.sz = s3[2];
    return 0;
}
}  // namespace
extern "C" {

int physad_deep_tangent_loss_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, float t, double* acc,
                                 float* Rs, float* Rx, float* Ry, float* Rz, void* stream) {
    if (!c || !acc) return fail(PHYSAD_E_INVALID, "deep_tangent_loss: null argument");
    if (int rc = check_residual_outputs(Rs, Rx, Ry, Rz, "deep_tangent_loss")) return rc;
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "deep_tangent_loss")) return rc;
    // one hidden layer: the one-hidden-layer analytic loss (its Jacobian products are precomputed on the host)
    if (c->deep_layers == 1 && c->deep_mode == 0) return physad_tangent_loss_dev(c, g, slab, t, acc, Rs, Rx, Ry, Rz, stream);
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    DeepTangentArgs a{};
    long long npts = 0;
    if (int rc = deep_tangent_args(c, g, slab, t, "deep_tangent_loss", a, &npts, st)) return rc;
    if (npts == 0) return zero_result(acc, 2, nullptr, 0, st);
    a.R[0] = Rs; a.R[1] = Rx; a.R[2] = Ry; a.R[3] = Rz;
    const int H = c->cfg.H;
    const int blocks = deep_tangent_blocks(H, npts, c->sm_count);
    if (int rc = ensure_grad_partials(c, size_t(blocks) * 2)) return rc;
    a.partials = c->gpart;
    CU(cudaError_t(deep_tangent_launch(H, false, a, blocks, acc, nullptr, st)));
    c->launches += 2;
    return 0;
}

int physad_deep_tangent_loss_grad_dev(physad_ctx* c, const physad_grid* g, const physad_slab* slab, const physad_phys_weights* w,
                                      float t, double* acc, double* grad, void* stream) {
    if (!c || !w || !acc || !grad) return fail(PHYSAD_E_INVALID, "deep_tangent_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "deep_tangent_loss_grad")) return rc;
    // one hidden layer: the one-hidden-layer closed loop, whose gradient layout is the same
    if (c->deep_layers == 1 && c->deep_mode == 0) return physad_tangent_loss_grad_dev(c, g, slab, w, t, acc, grad, stream);
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    DeepTangentArgs a{};
    long long npts = 0;
    if (int rc = deep_tangent_args(c, g, slab, t, "deep_tangent_loss_grad", a, &npts, st)) return rc;
    const int H = c->cfg.H, L = c->deep_layers;
    const size_t P = deep_grad_len(H, L);
    if (npts == 0) return zero_result(acc, 2, grad, P, st);
    vjp_scales(g, w, &a.scale_s, &a.scale_u);   // 2 w / float(N) of the whole grid: slab results add up to the grid's
    const int blocks = deep_tangent_blocks(H, npts, c->sm_count);
    if (int rc = grow(c->dckpt, c->dckpt_cap, size_t(blocks) * deep_tangent_ckpt_floats(L))) return rc;
    if (int rc = ensure_grad_partials(c, size_t(blocks) * (P + 2))) return rc;
    a.ckpt = c->dckpt;
    a.partials = c->gpart;
    CU(cudaError_t(deep_tangent_launch(H, true, a, blocks, acc, grad, st)));
    c->launches += 2;
    return 0;
}

int physad_deep_tangent_loss_grad_host(physad_ctx* c, const physad_grid* g, const physad_phys_weights* w, float t,
                                       float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dWh, float* dbh,
                                       float* dW2, float* db2) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "deep_tangent_loss_grad: null argument");
    if (int rc = check_grid(g)) return rc;
    if (int rc = deep_ready(c, "deep_tangent_loss_grad")) return rc;
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    if (int rc = physad_deep_tangent_loss_grad_dev(c, g, nullptr, w, t, c->d_dgrad, c->d_dgrad + 2, c->stream)) return rc;
    return grad_to_host(c, 2, size_t(g->nx) * g->ny * g->nz, w, loss_sigma, loss_u, {dW1, db1, dWh, dbh, dW2, db2});
}

// ---- deeper networks at caller-supplied points: forward and data-fit loss + gradient (deep_data_kernels.cuh) --------
}  // extern "C"  (helpers below)
namespace {
template <int H>
int launch_deep_points(physad_ctx* c, const DeepArgs& a, cudaStream_t st) {
    MlpConst<H> k;
    const float no_t[3] = {0.f, 0.f, 0.f};   // points mode forms W1[h,3] * t per row; the pre-rounded products are unused
    fill_const<H>(c, no_t, k);
    CU(cudaError_t(deep_points_launch(H, &k, a, c->sm_count, st)));
    c->launches++;
    return 0;
}

// how the kernel of deep_data_body.cuh forms its seeds: data fit, matched pairs, or the caller's cotangents (the VJP)
enum class DataSeeds { data, pairs, vjp };

template <int H>
int launch_deep_data(physad_ctx* c, DataSeeds seeds, const DeepDataArgs& a, int blocks, double* grad, double* acc, cudaStream_t st) {
    MlpConst<H> k;
    const float no_t[3] = {0.f, 0.f, 0.f};   // only the output pairs w2 / b2 are read
    fill_const<H>(c, no_t, k);
    CU(cudaError_t(seeds == DataSeeds::pairs ? deep_pair_launch(H, &k, a, blocks, grad, acc, st)
                   : seeds == DataSeeds::vjp ? vjp_points_launch(H, &k, a, blocks, grad, acc, st)
                                             : deep_data_launch(H, &k, a, blocks, grad, acc, st)));
    c->launches += 2;
    return 0;
}

// checks shared by the forward and the data loss at points: deep weights, strict mode
int deep_points_ready(const physad_ctx* c, const char* what) {
    if (int rc = deep_ready(c, what)) return rc;
    if (c->deep_mode != 0)
        return fail(PHYSAD_E_UNSUPPORTED, std::string(what) + ": strict fp32 only (set_deep_mode(0))");
    return 0;
}

bool misaligned16(const void* p) { return uintptr_t(p) % 16 != 0; }
}  // namespace
extern "C" {

int physad_mlp_forward_deep_dev(physad_ctx* c, const float* x, float* y, size_t B, void* stream) {
    if (!c) return fail(PHYSAD_E_INVALID, "mlp_forward_deep: null context");
    if (int rc = deep_points_ready(c, "mlp_forward_deep")) return rc;
    if (B && (!x || !y)) return fail(PHYSAD_E_INVALID, "mlp_forward_deep: null argument");
    if (B && (misaligned16(x) || misaligned16(y))) return fail(PHYSAD_E_INVALID, "mlp_forward_deep: x and y must be 16-byte aligned");
    if (B == 0) return 0;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    DeepArgs a{};
    a.hidden_layers = c->deep_layers;
    a.W1 = c->dW1; a.b1 = c->db1; a.wh = c->d_wh; a.bh = c->d_bh;
    a.pts = reinterpret_cast<const float4*>(x);
    a.n_points = (long long)B;
    a.out_aos = reinterpret_cast<float4*>(y);
    switch (c->cfg.H) {
        case 32: return launch_deep_points<32>(c, a, st);
        case 64: return launch_deep_points<64>(c, a, st);
        default: return launch_deep_points<128>(c, a, st);
    }
}

int physad_mlp_forward_deep_host(physad_ctx* c, const float* x, float* y, size_t B) {
    if (!c) return fail(PHYSAD_E_INVALID, "mlp_forward_deep: null context");
    if (int rc = deep_points_ready(c, "mlp_forward_deep")) return rc;
    if (B && (!x || !y)) return fail(PHYSAD_E_INVALID, "mlp_forward_deep: null argument");
    if (B == 0) return 0;
    DeviceGuard dg(c->device);
    Staged a[2] = {{x, nullptr, B * 4 * sizeof(float)}, {nullptr, y, B * 4 * sizeof(float)}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_forward_deep_dev(c, a[0].dev, a[1].dev, B, c->stream)) return rc;
    return stage_out(c, a);
}

}  // extern "C"  (helpers below)
namespace {
// lam[4] of the fit losses (data, pair, derivative): NULL gives 1/4 each (the mean over the four outputs); each must be
// finite and non-negative
int read_lam(const float* lam, float lw[4], const std::string& what) {
    for (int o = 0; o < 4; ++o) lw[o] = 0.25f;
    if (lam) {
        for (int o = 0; o < 4; ++o) {
            if (!std::isfinite(lam[o]) || lam[o] < 0.f) return fail(PHYSAD_E_INVALID, what + ": lam must be finite and non-negative");
            lw[o] = lam[o];
        }
    }
    return 0;
}

// The launch shared by the data loss, the pair loss and the VJP at a.n > 0 rows: the weights, the grid, the checkpoint, the
// partials, the kernel and the reduction.  `a` brings the rows and the seed inputs; the network's fields are filled here.
// acc null (the VJP): the reduction's (zero) loss sum goes to a slot after the partials.
int deep_data_run(physad_ctx* c, DataSeeds seeds, DeepDataArgs& a, double* grad, double* acc, cudaStream_t st) {
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    const int H = c->cfg.H, L = c->deep_layers;
    const size_t P = deep_grad_len(H, L);
    const int blocks = deep_data_blocks(H, a.n, c->sm_count);
    if (int rc = grow(c->dckpt, c->dckpt_cap, size_t(blocks) * deep_data_ckpt_floats(H, L))) return rc;
    const size_t np = size_t(blocks) * (P + 1);
    if (int rc = ensure_grad_partials(c, np + (acc ? 0 : 1))) return rc;
    a.hidden_layers = L;
    a.W1 = c->dW1; a.b1 = c->db1; a.W2 = c->dW2;
    a.wh = c->d_wh; a.bh = c->d_bh;
    a.ckpt = c->dckpt;
    a.partials = c->gpart;
    if (!acc) acc = c->gpart + np;
    switch (H) {
        case 32: return launch_deep_data<32>(c, seeds, a, blocks, grad, acc, st);
        case 64: return launch_deep_data<64>(c, seeds, a, blocks, grad, acc, st);
        default: return launch_deep_data<128>(c, seeds, a, blocks, grad, acc, st);
    }
}

// The data loss (B points and their targets) and the pair loss (B pairs = 2B rows of x, no target) share everything but
// the kernel: the checks, the scratch, the arguments and the reduction.  `what` names the caller in error messages.
int deep_fit_dev(physad_ctx* c, const char* what, bool pairs, const float* x, const float* target, size_t B, const float* lam,
                 size_t n_norm, double* acc, double* grad, void* stream) {
    const std::string w(what);
    if (!c) return fail(PHYSAD_E_INVALID, w + ": null context");
    if (int rc = deep_points_ready(c, what)) return rc;
    if (!acc || !grad || (B && (!x || (!pairs && !target)))) return fail(PHYSAD_E_INVALID, w + ": null argument");
    if (B && (misaligned16(x) || (!pairs && misaligned16(target))))
        return fail(PHYSAD_E_INVALID, w + (pairs ? ": x must be 16-byte aligned" : ": x and target must be 16-byte aligned"));
    if (uintptr_t(acc) % 8 || uintptr_t(grad) % 8) return fail(PHYSAD_E_INVALID, w + ": acc and grad must be 8-byte aligned");
    if (n_norm == 0) return fail(PHYSAD_E_INVALID, w + ": n_norm must be positive");
    float lw[4];
    if (int rc = read_lam(lam, lw, w)) return rc;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    const int H = c->cfg.H, L = c->deep_layers;
    const size_t P = deep_grad_len(H, L);
    if (B == 0) return zero_result(acc, 1, grad, P, st);   // an empty shard: zero sum, zero gradient
    DeepDataArgs a{};
    a.n = (long long)(pairs ? 2 * B : B);
    a.x = reinterpret_cast<const float4*>(x);
    a.target = reinterpret_cast<const float4*>(target);
    for (int o = 0; o < 4; ++o) {
        a.coef[o] = float(2.0 * double(lw[o]) / double(n_norm));
        a.lam[o] = double(lw[o]);
    }
    return deep_data_run(c, pairs ? DataSeeds::pairs : DataSeeds::data, a, grad, acc, st);
}

// The host forms: x (and target) uploaded, n_norm = B, the gradient split into set_weights_deep's six arrays.
int deep_fit_host(physad_ctx* c, const char* what, bool pairs, const float* x, const float* target, size_t B, const float* lam,
                  float* loss, float* dW1, float* db1, float* dWh, float* dbh, float* dW2, float* db2) {
    if (!c) return fail(PHYSAD_E_INVALID, std::string(what) + ": null context");
    if (int rc = deep_points_ready(c, what)) return rc;
    if (B && (!x || (!pairs && !target))) return fail(PHYSAD_E_INVALID, std::string(what) + ": null argument");
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    const size_t bytes = B * (pairs ? 8 : 4) * sizeof(float);
    Staged a[2] = {{x, nullptr, bytes}, {target, nullptr, pairs ? 0 : bytes}};
    if (int rc = stage_in(c, a)) return rc;
    // n_norm = B; an empty set (B = 0) gives a zero loss and a zero gradient
    const size_t n = B ? B : 1;
    if (int rc = deep_fit_dev(c, what, pairs, a[0].dev, pairs ? nullptr : a[1].dev, B, lam, n, c->d_dgrad, c->d_dgrad + 1, c->stream))
        return rc;
    return grad_to_host(c, 1, n, nullptr, loss, nullptr, {dW1, db1, dWh, dbh, dW2, db2});
}
}  // namespace
extern "C" {

int physad_deep_data_loss_grad_dev(physad_ctx* c, const float* x, const float* target, size_t B, const float* lam,
                                   size_t n_norm, double* acc, double* grad, void* stream) {
    return deep_fit_dev(c, "deep_data_loss_grad", false, x, target, B, lam, n_norm, acc, grad, stream);
}

int physad_deep_data_loss_grad_host(physad_ctx* c, const float* x, const float* target, size_t B, const float* lam,
                                    float* loss, float* dW1, float* db1, float* dWh, float* dbh, float* dW2, float* db2) {
    return deep_fit_host(c, "deep_data_loss_grad", false, x, target, B, lam, loss, dW1, db1, dWh, dbh, dW2, db2);
}

// ---- periodic boundaries at points: the matched-pair loss of deeper networks (deep_data_kernels.cuh) -------------------
int physad_deep_pair_loss_grad_dev(physad_ctx* c, const float* x, size_t B, const float* lam, size_t n_norm, double* acc,
                                   double* grad, void* stream) {
    return deep_fit_dev(c, "deep_pair_loss_grad", true, x, nullptr, B, lam, n_norm, acc, grad, stream);
}

int physad_deep_pair_loss_grad_host(physad_ctx* c, const float* x, size_t B, const float* lam, float* loss, float* dW1,
                                    float* db1, float* dWh, float* dbh, float* dW2, float* db2) {
    return deep_fit_host(c, "deep_pair_loss_grad", true, x, nullptr, B, lam, loss, dW1, db1, dWh, dbh, dW2, db2);
}

// ---- analytic loss of deeper networks at caller-supplied points (collocation points; deep_tangent_kernels.cuh) ---------
int physad_grid_input_scales(const physad_grid* g, int norm, float dcdx[3]) {
    if (!g || !dcdx) return fail(PHYSAD_E_INVALID, "grid_input_scales: null argument");
    if (g->nx <= 0 || g->ny <= 0 || g->nz <= 0) return fail(PHYSAD_E_INVALID, "grid_input_scales: grid extents must be positive");
    if (norm != 0 && norm != 1) return fail(PHYSAD_E_INVALID, "grid_input_scales: norm must be 0 (ZeroToOne) or 1 (MinusOneToOne)");
    input_scales(g, norm, dcdx);
    return 0;
}

}  // extern "C"  (helpers below)
namespace {
// checks shared by the points loss and the points loss + gradient call
int colloc_check(const float* x, size_t B, const float* dcdx, const char* what) {
    if (B && !x) return fail(PHYSAD_E_INVALID, std::string(what) + ": null argument");
    if (B && misaligned16(x)) return fail(PHYSAD_E_INVALID, std::string(what) + ": x must be 16-byte aligned");
    for (int k = 0; k < 3; ++k)
        if (!std::isfinite(dcdx[k])) return fail(PHYSAD_E_INVALID, std::string(what) + ": dcdx must be finite");
    return 0;
}

// the kernel arguments of B > 0 points; uploads the context's weights first (that may move the device buffers).  dcdx
// null: the derivative calls, which read no space scales
int colloc_args(physad_ctx* c, const float* x, size_t B, const float* dcdx, DeepTangentArgs& a, cudaStream_t st) {
    if (int rc = upload_weights_if_stale(c, st)) return rc;
    a.hidden_layers = c->deep_layers;
    a.W1 = c->dW1; a.b1 = c->db1; a.W2 = c->dW2; a.b2 = c->db2;
    a.wh = c->d_wh; a.bh = c->d_bh;
    if (dcdx) { a.sx = dcdx[0]; a.sy = dcdx[1]; a.sz = dcdx[2]; }
    a.pts = reinterpret_cast<const float4*>(x);
    a.n_points = (long long)B;
    return 0;
}

// how the points kernel of deep_tangent_body.cuh forms its seeds: physics residuals, derivative fit, or the caller's
// cotangents (the VJP)
enum class TangentSeeds { physics, deriv, vjp };

// The gradient launch at B > 0 points, shared by the physics loss (k_colloc_tangent), the derivative-fit loss
// (k_deriv_tangent) and the VJP (k_vjp_tangent): one kernel body, so one scratch, L x 80 KB of checkpoint and P + 2
// partials per block.  The physics loss returns both sums in acc[2]; the derivative loss one and the VJP none, so their
// reductions write two doubles after the partials and acc (if any) is copied out from there.
int colloc_grad_launch(physad_ctx* c, TangentSeeds seeds, DeepTangentArgs& a, double* acc, double* grad, cudaStream_t st) {
    const int H = c->cfg.H, L = c->deep_layers;
    const size_t P = deep_grad_len(H, L);
    const int blocks = deep_tangent_blocks(H, a.n_points, c->sm_count);
    if (int rc = grow(c->dckpt, c->dckpt_cap, size_t(blocks) * deep_tangent_ckpt_floats(L))) return rc;
    const size_t np = size_t(blocks) * (P + 2);
    const bool physics = seeds == TangentSeeds::physics;
    if (int rc = ensure_grad_partials(c, np + (physics ? 0 : 2))) return rc;
    a.ckpt = c->dckpt;
    a.partials = c->gpart;
    if (physics) {
        CU(cudaError_t(colloc_tangent_launch(H, true, a, blocks, acc, grad, st)));
    } else {
        CU(cudaError_t(seeds == TangentSeeds::deriv ? deriv_tangent_launch(H, true, a, blocks, c->gpart + np, grad, st)
                                                    : vjp_tangent_launch(H, a, blocks, c->gpart + np, grad, st)));
        if (acc) CU(cudaMemcpyAsync(acc, c->gpart + np, sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    c->launches += 2;
    return 0;
}
}  // namespace
extern "C" {

int physad_deep_tangent_points_loss_dev(physad_ctx* c, const float* x, size_t B, const float* dcdx, double* acc, float* R,
                                        void* stream) {
    if (!c) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss: null context");
    if (int rc = deep_points_ready(c, "deep_tangent_points_loss")) return rc;
    if (!acc || !dcdx) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss: null argument");
    if (uintptr_t(acc) % 8) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss: acc must be 8-byte aligned");
    if (R && misaligned16(R)) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss: R must be 16-byte aligned");
    if (int rc = colloc_check(x, B, dcdx, "deep_tangent_points_loss")) return rc;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (B == 0) return zero_result(acc, 2, nullptr, 0, st);
    DeepTangentArgs a{};
    if (int rc = colloc_args(c, x, B, dcdx, a, st)) return rc;
    a.R_pts = reinterpret_cast<float4*>(R);
    const int H = c->cfg.H;
    const int blocks = deep_tangent_blocks(H, (long long)B, c->sm_count);
    if (int rc = ensure_grad_partials(c, size_t(blocks) * 2)) return rc;
    a.partials = c->gpart;
    CU(cudaError_t(colloc_tangent_launch(H, false, a, blocks, acc, nullptr, st)));
    c->launches += 2;
    return 0;
}

int physad_deep_tangent_points_loss_grad_dev(physad_ctx* c, const float* x, size_t B, const float* dcdx,
                                             const physad_phys_weights* w, size_t n_norm, double* acc, double* grad,
                                             void* stream) {
    if (!c) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss_grad: null context");
    if (int rc = deep_points_ready(c, "deep_tangent_points_loss_grad")) return rc;
    if (!w || !acc || !grad || !dcdx) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss_grad: null argument");
    if (uintptr_t(acc) % 8 || uintptr_t(grad) % 8)
        return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss_grad: acc and grad must be 8-byte aligned");
    if (n_norm == 0) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss_grad: n_norm must be positive");
    if (int rc = colloc_check(x, B, dcdx, "deep_tangent_points_loss_grad")) return rc;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    const int H = c->cfg.H, L = c->deep_layers;
    const size_t P = deep_grad_len(H, L);
    if (B == 0) return zero_result(acc, 2, grad, P, st);   // an empty shard: zero sums, zero gradient
    DeepTangentArgs a{};
    if (int rc = colloc_args(c, x, B, dcdx, a, st)) return rc;
    // vjp_scales' formula with n_norm for N: shards with the same n_norm add up to the whole set's gradient
    a.scale_s = 2.f * w->w_sigma / float(n_norm);
    a.scale_u = 2.f * w->w_u / float(n_norm);
    return colloc_grad_launch(c, TangentSeeds::physics, a, acc, grad, st);
}

int physad_deep_tangent_points_loss_grad_host(physad_ctx* c, const float* x, size_t B, const float* dcdx,
                                              const physad_phys_weights* w, float* loss_sigma, float* loss_u, float* dW1,
                                              float* db1, float* dWh, float* dbh, float* dW2, float* db2) {
    if (!c) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss_grad: null context");
    if (int rc = deep_points_ready(c, "deep_tangent_points_loss_grad")) return rc;
    if (!w || !dcdx || (B && !x)) return fail(PHYSAD_E_INVALID, "deep_tangent_points_loss_grad: null argument");
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    Staged a[1] = {{x, nullptr, B * 4 * sizeof(float)}};
    if (int rc = stage_in(c, a)) return rc;
    // n_norm = B; an empty set (B = 0) gives zero losses and a zero gradient
    const size_t n = B ? B : 1;
    if (int rc = physad_deep_tangent_points_loss_grad_dev(c, a[0].dev, B, dcdx, w, n, c->d_dgrad, c->d_dgrad + 2, c->stream))
        return rc;
    return grad_to_host(c, 2, n, w, loss_sigma, loss_u, {dW1, db1, dWh, dbh, dW2, db2});
}

// ---- Neumann boundaries at points: the Jacobian of deeper networks and the derivative-fit loss (deep_tangent_kernels.cuh)
int physad_mlp_jacobian_deep_dev(physad_ctx* c, const float* x, float* y, float* J, size_t B, void* stream) {
    if (!c) return fail(PHYSAD_E_INVALID, "mlp_jacobian_deep: null context");
    if (int rc = deep_points_ready(c, "mlp_jacobian_deep")) return rc;
    if (B && (!x || !y || !J)) return fail(PHYSAD_E_INVALID, "mlp_jacobian_deep: null argument");
    if (B && (misaligned16(x) || misaligned16(y) || misaligned16(J)))
        return fail(PHYSAD_E_INVALID, "mlp_jacobian_deep: x, y and J must be 16-byte aligned");
    if (B == 0) return 0;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    DeepTangentArgs a{};
    if (int rc = colloc_args(c, x, B, nullptr, a, st)) return rc;
    a.y_pts = reinterpret_cast<float4*>(y);
    a.J_pts = reinterpret_cast<float4*>(J);
    const int H = c->cfg.H;
    CU(cudaError_t(deriv_tangent_launch(H, false, a, deep_tangent_blocks(H, (long long)B, c->sm_count), nullptr, nullptr, st)));
    c->launches++;
    return 0;
}

int physad_mlp_jacobian_deep_host(physad_ctx* c, const float* x, float* y, float* J, size_t B) {
    if (!c) return fail(PHYSAD_E_INVALID, "mlp_jacobian_deep: null context");
    if (int rc = deep_points_ready(c, "mlp_jacobian_deep")) return rc;
    if (B && (!x || !y || !J)) return fail(PHYSAD_E_INVALID, "mlp_jacobian_deep: null argument");
    if (B == 0) return 0;
    DeviceGuard dg(c->device);
    const size_t bytes = B * 4 * sizeof(float);
    Staged a[3] = {{x, nullptr, bytes}, {nullptr, y, bytes}, {nullptr, J, 4 * bytes}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_jacobian_deep_dev(c, a[0].dev, a[1].dev, a[2].dev, B, c->stream)) return rc;
    return stage_out(c, a);
}

int physad_deep_deriv_loss_grad_dev(physad_ctx* c, const float* x, const float* dir, const float* target, size_t B,
                                    const float* lam, size_t n_norm, double* acc, double* grad, void* stream) {
    const std::string w("deep_deriv_loss_grad");
    if (!c) return fail(PHYSAD_E_INVALID, w + ": null context");
    if (int rc = deep_points_ready(c, w.c_str())) return rc;
    if (!acc || !grad || (B && (!x || !dir || !target))) return fail(PHYSAD_E_INVALID, w + ": null argument");
    if (B && (misaligned16(x) || misaligned16(dir) || misaligned16(target)))
        return fail(PHYSAD_E_INVALID, w + ": x, dir and target must be 16-byte aligned");
    if (uintptr_t(acc) % 8 || uintptr_t(grad) % 8) return fail(PHYSAD_E_INVALID, w + ": acc and grad must be 8-byte aligned");
    if (n_norm == 0) return fail(PHYSAD_E_INVALID, w + ": n_norm must be positive");
    float lw[4];
    if (int rc = read_lam(lam, lw, w)) return rc;
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (B == 0) return zero_result(acc, 1, grad, deep_grad_len(c->cfg.H, c->deep_layers), st);   // an empty shard
    DeepTangentArgs a{};
    if (int rc = colloc_args(c, x, B, nullptr, a, st)) return rc;
    a.dirs = reinterpret_cast<const float4*>(dir);
    a.targets = reinterpret_cast<const float4*>(target);
    for (int o = 0; o < 4; ++o) {   // deep_fit_dev's coefficients: shards with the same n_norm add up
        a.coef[o] = float(2.0 * double(lw[o]) / double(n_norm));
        a.lam[o] = double(lw[o]);
    }
    return colloc_grad_launch(c, TangentSeeds::deriv, a, acc, grad, st);
}

int physad_deep_deriv_loss_grad_host(physad_ctx* c, const float* x, const float* dir, const float* target, size_t B,
                                     const float* lam, float* loss, float* dW1, float* db1, float* dWh, float* dbh, float* dW2,
                                     float* db2) {
    if (!c) return fail(PHYSAD_E_INVALID, "deep_deriv_loss_grad: null context");
    if (int rc = deep_points_ready(c, "deep_deriv_loss_grad")) return rc;
    if (B && (!x || !dir || !target)) return fail(PHYSAD_E_INVALID, "deep_deriv_loss_grad: null argument");
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    const size_t bytes = B * 4 * sizeof(float);
    Staged a[3] = {{x, nullptr, bytes}, {dir, nullptr, bytes}, {target, nullptr, bytes}};
    if (int rc = stage_in(c, a)) return rc;
    // n_norm = B; an empty set (B = 0) gives a zero loss and a zero gradient
    const size_t n = B ? B : 1;
    if (int rc = physad_deep_deriv_loss_grad_dev(c, a[0].dev, a[1].dev, a[2].dev, B, lam, n, c->d_dgrad, c->d_dgrad + 1, c->stream))
        return rc;
    return grad_to_host(c, 1, n, nullptr, loss, nullptr, {dW1, db1, dWh, dbh, dW2, db2});
}

// ---- vector-Jacobian products of deeper networks at points (deep_data_kernels.cuh, deep_tangent_kernels.cuh) ----------
int physad_mlp_vjp_deep_dev(physad_ctx* c, const float* x, const float* ybar, size_t B, double* grad, void* stream) {
    const std::string w("mlp_vjp_deep");
    if (!c) return fail(PHYSAD_E_INVALID, w + ": null context");
    if (int rc = deep_points_ready(c, w.c_str())) return rc;
    if (!grad || (B && (!x || !ybar))) return fail(PHYSAD_E_INVALID, w + ": null argument");
    if (B && (misaligned16(x) || misaligned16(ybar))) return fail(PHYSAD_E_INVALID, w + ": x and ybar must be 16-byte aligned");
    if (uintptr_t(grad) % 8) return fail(PHYSAD_E_INVALID, w + ": grad must be 8-byte aligned");
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (B == 0) return zero_result(nullptr, 0, grad, deep_grad_len(c->cfg.H, c->deep_layers), st);   // an empty shard
    DeepDataArgs a{};
    a.n = (long long)B;
    a.x = reinterpret_cast<const float4*>(x);
    a.ybar = reinterpret_cast<const float4*>(ybar);
    return deep_data_run(c, DataSeeds::vjp, a, grad, nullptr, st);
}

int physad_mlp_vjp_deep_host(physad_ctx* c, const float* x, const float* ybar, size_t B, float* dW1, float* db1, float* dWh,
                             float* dbh, float* dW2, float* db2) {
    if (!c) return fail(PHYSAD_E_INVALID, "mlp_vjp_deep: null context");
    if (int rc = deep_points_ready(c, "mlp_vjp_deep")) return rc;
    if (B && (!x || !ybar)) return fail(PHYSAD_E_INVALID, "mlp_vjp_deep: null argument");
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    Staged a[2] = {{x, nullptr, B * 4 * sizeof(float)}, {ybar, nullptr, B * 4 * sizeof(float)}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_vjp_deep_dev(c, a[0].dev, a[1].dev, B, c->d_dgrad, c->stream)) return rc;
    return grad_to_host(c, 0, 0, nullptr, nullptr, nullptr, {dW1, db1, dWh, dbh, dW2, db2});
}

int physad_mlp_jacobian_vjp_deep_dev(physad_ctx* c, const float* x, const float* ybar, const float* Jbar, size_t B, double* grad,
                                     void* stream) {
    const std::string w("mlp_jacobian_vjp_deep");
    if (!c) return fail(PHYSAD_E_INVALID, w + ": null context");
    if (int rc = deep_points_ready(c, w.c_str())) return rc;
    if (!grad || (B && (!x || !ybar || !Jbar))) return fail(PHYSAD_E_INVALID, w + ": null argument");
    if (B && (misaligned16(x) || misaligned16(ybar) || misaligned16(Jbar)))
        return fail(PHYSAD_E_INVALID, w + ": x, ybar and Jbar must be 16-byte aligned");
    if (uintptr_t(grad) % 8) return fail(PHYSAD_E_INVALID, w + ": grad must be 8-byte aligned");
    DeviceGuard dg(c->device);
    cudaStream_t st = cudaStream_t(stream);
    if (B == 0) return zero_result(nullptr, 0, grad, deep_grad_len(c->cfg.H, c->deep_layers), st);   // an empty shard
    DeepTangentArgs a{};
    if (int rc = colloc_args(c, x, B, nullptr, a, st)) return rc;
    a.ybar = reinterpret_cast<const float4*>(ybar);
    a.Jbar = reinterpret_cast<const float4*>(Jbar);
    return colloc_grad_launch(c, TangentSeeds::vjp, a, nullptr, grad, st);
}

int physad_mlp_jacobian_vjp_deep_host(physad_ctx* c, const float* x, const float* ybar, const float* Jbar, size_t B, float* dW1,
                                      float* db1, float* dWh, float* dbh, float* dW2, float* db2) {
    if (!c) return fail(PHYSAD_E_INVALID, "mlp_jacobian_vjp_deep: null context");
    if (int rc = deep_points_ready(c, "mlp_jacobian_vjp_deep")) return rc;
    if (B && (!x || !ybar || !Jbar)) return fail(PHYSAD_E_INVALID, "mlp_jacobian_vjp_deep: null argument");
    DeviceGuard dg(c->device);
    if (int rc = ensure_host_grad(c)) return rc;
    const size_t bytes = B * 4 * sizeof(float);
    Staged a[3] = {{x, nullptr, bytes}, {ybar, nullptr, bytes}, {Jbar, nullptr, 4 * bytes}};
    if (int rc = stage_in(c, a)) return rc;
    if (int rc = physad_mlp_jacobian_vjp_deep_dev(c, a[0].dev, a[1].dev, a[2].dev, B, c->d_dgrad, c->stream)) return rc;
    return grad_to_host(c, 0, 0, nullptr, nullptr, nullptr, {dW1, db1, dWh, dbh, dW2, db2});
}

int physad_plan_ranges(int tiles, int planes, int slots, int* out, int out_cap) {
    if (tiles < 1 || planes < 1 || slots < 1 || !out) return fail(PHYSAD_E_INVALID, "plan_ranges: bad argument");
    const std::vector<int> r = balanced_ranges(tiles, planes, std::min<long long>(slots, (long long)tiles * planes), 0.9);
    if (int(r.size()) > out_cap) return fail(PHYSAD_E_INVALID, "plan_ranges: output too small");
    std::copy(r.begin(), r.end(), out);
    return int(r.size());
}

int physad_xchg_export(physad_ctx* c, void* handle_out) {
    if (!c || !handle_out) return fail(PHYSAD_E_INVALID, "xchg_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == PHYSAD_XCHG_HANDLE_BYTES, "IPC handle size");
    DeviceGuard dg(c->device);
    if (!c->xbuf) {
        CU(cudaMalloc(&c->xbuf, 2 * XCHG_MAX_RANKS * sizeof(XSlot)));
        CU(cudaMemset(c->xbuf, 0, 2 * XCHG_MAX_RANKS * sizeof(XSlot)));
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, c->xbuf));
    std::memcpy(handle_out, &h, sizeof(h));
    return 0;
}

int physad_xchg_connect(physad_ctx* c, int rank, int world, const void* handles) {
    if (!c || !handles) return fail(PHYSAD_E_INVALID, "xchg_connect: null argument");
    if (world < 1 || world > XCHG_MAX_RANKS || rank < 0 || rank >= world)
        return fail(PHYSAD_E_UNSUPPORTED, "xchg_connect: 1 <= world <= 8 ranks of one node");
    if (!c->xbuf) return fail(PHYSAD_E_INVALID, "xchg_connect: call physad_xchg_export first");
    DeviceGuard dg(c->device);
    physad_xchg_disconnect(c);
    for (int p = 0; p < world; ++p) {
        if (p == rank) { c->xpeer[p] = c->xbuf; continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, static_cast<const char*>(handles) + size_t(p) * sizeof(h), sizeof(h));
        void* ptr = nullptr;
        CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        c->xpeer[p] = static_cast<XSlot*>(ptr);
    }
    CU(cudaMemset(c->xbuf, 0, 2 * XCHG_MAX_RANKS * sizeof(XSlot)));
    CU(cudaDeviceSynchronize());
    c->xrank = rank; c->xworld = world; c->xepoch = 0;
    return 0;
}

int physad_xchg_disconnect(physad_ctx* c) {
    if (!c) return 0;
    for (int p = 0; p < XCHG_MAX_RANKS; ++p) {
        if (c->xpeer[p] && c->xpeer[p] != c->xbuf) cudaIpcCloseMemHandle(c->xpeer[p]);
        c->xpeer[p] = nullptr;
    }
    c->xworld = 1; c->xrank = 0; c->xepoch = 0;
    return 0;
}

namespace {
// Wait for the fused kernel's last block to publish sequence number `seq` in the mapped host record.  Spins on
// host memory (the record is written once per step over PCIe); every few microseconds the stream is queried
// so that a failed launch or a dead device turns into an error instead of a hang.
int wait_host_result(physad_ctx* c, unsigned long long seq, double acc[2]) {
    HostResult* r = c->h_res;
    int done_polls = 0;
    for (unsigned spins = 1;; ++spins) {
        if (__atomic_load_n(&r->seq, __ATOMIC_ACQUIRE) == seq) break;
        if ((spins & 0x3ff) == 0) {
            const cudaError_t e = cudaStreamQuery(c->stream);
            if (e != cudaSuccess && e != cudaErrorNotReady)
                return fail(int(e), std::string("fused kernel failed: ") + cudaGetErrorString(e));
            if (e == cudaSuccess && ++done_polls > 1000)
                return fail(PHYSAD_E_INVALID, "fused kernel finished without publishing its result");
        }
    }
    acc[0] = r->a;
    acc[1] = r->b;
    if (r->status != 0) return fail(PHYSAD_E_PEER_TIMEOUT, "in-kernel exchange: a peer rank never arrived (sums are NaN)");
    return 0;
}
}  // namespace

int physad_fused_loss_host(physad_ctx* c, const physad_grid* g, const physad_mlp_config* cfg, const float* W1,
                           const float* b1, const float* W2, const float* b2, const physad_phys_weights* w, float t,
                           float dt, float* loss_sigma, float* loss_u, float* Rs, float* Rx, float* Ry, float* Rz) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "fused_loss: null argument");
    if (int rc = check_grid(g)) return rc;
    if (cfg) {
        if (int rc = physad_set_weights(c, cfg, W1, b1, W2, b2)) return rc;
    }
    DeviceGuard dg(c->device);
    const size_t N = size_t(g->nx) * g->ny * g->nz;
    float* host_r[4] = {Rs, Rx, Ry, Rz};
    const bool want_r = Rs || Rx || Ry || Rz;
    float* r = nullptr;
    if (want_r) {
        if (int rc = ensure_scratch(c, 4 * N * sizeof(float))) return rc;
        r = reinterpret_cast<float*>(c->scratch);
    }
    if (!want_r) {   // 16-byte result: straight into mapped host memory, no copy, no stream sync
        c->want_host_seq = ++c->res_seq;
        const int rc = physad_fused_loss_dev(c, g, nullptr, t, dt, c->d_acc, nullptr, nullptr, nullptr, nullptr, c->stream);
        const unsigned long long seq = c->want_host_seq;
        c->want_host_seq = 0;
        if (rc) return rc;
        double acc[2];
        if (int rc2 = wait_host_result(c, seq, acc)) return rc2;
        physad_finalize_loss(acc, w, N, loss_sigma, loss_u);
        return 0;
    }
    if (int rc = physad_fused_loss_dev(c, g, nullptr, t, dt, c->d_acc, r, r ? r + N : nullptr, r ? r + 2 * N : nullptr,
                                       r ? r + 3 * N : nullptr, c->stream))
        return rc;
    CU(cudaMemcpyAsync(c->h_acc, c->d_acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    for (int k = 0; k < 4; ++k)
        if (host_r[k]) CU(cudaMemcpyAsync(host_r[k], r + k * N, N * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    physad_finalize_loss(c->h_acc, w, N, loss_sigma, loss_u);
    return 0;
}

int physad_fused_loss_slab_host(physad_ctx* c, const physad_grid* g, const physad_slab* slab, const physad_mlp_config* cfg,
                                const float* W1, const float* b1, const float* W2, const float* b2,
                                const physad_phys_weights* w, float t, float dt, int exchange, float* loss_sigma,
                                float* loss_u) {
    if (!c || !w) return fail(PHYSAD_E_INVALID, "fused_loss_slab: null argument");
    if (int rc = check_grid(g)) return rc;
    if (cfg) {
        if (int rc = physad_set_weights(c, cfg, W1, b1, W2, b2)) return rc;
    }
    DeviceGuard dg(c->device);
    // the kernel's last block writes {sums, status, seq} straight into mapped pinned host memory; poll it
    c->want_host_seq = ++c->res_seq;
    const int rc = exchange ? physad_fused_loss_allreduce_dev(c, g, slab, t, dt, c->d_acc, nullptr, nullptr, nullptr, nullptr, c->stream)
                            : physad_fused_loss_dev(c, g, slab, t, dt, c->d_acc, nullptr, nullptr, nullptr, nullptr, c->stream);
    const unsigned long long seq = c->want_host_seq;
    c->want_host_seq = 0;
    if (rc) return rc;
    double acc[2];
    if (int rc2 = wait_host_result(c, seq, acc)) return rc2;
    physad_finalize_loss(acc, w, size_t(g->nx) * g->ny * g->nz, loss_sigma, loss_u);
    return 0;
}

int physad_xchg_status(physad_ctx* c, int* timed_out) {
    if (!c || !timed_out) return fail(PHYSAD_E_INVALID, "xchg_status: null argument");
    DeviceGuard dg(c->device);
    unsigned int v = 0;
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(&v, c->d_status, sizeof(v), cudaMemcpyDeviceToHost));
    if (v) CU(cudaMemset(c->d_status, 0, sizeof(v)));
    *timed_out = v ? 1 : 0;
    return 0;
}

int physad_set_fused_trace(physad_ctx* c, unsigned long long* dev_buf, int blocks_cap) {
    if (!c) return fail(PHYSAD_E_INVALID, "set_fused_trace: null context");
    c->trace = dev_buf;
    c->trace_blocks = dev_buf ? blocks_cap : 0;
    return 0;
}

void physad_finalize_loss(const double acc[2], const physad_phys_weights* w, size_t n_global, float* loss_sigma,
                          float* loss_u) {
    // src/phys_cpu.cpp:146-148 forms `double invN = 1.0 / double(N)` and MULTIPLIES: float(w * acc * invN)
    const double invN = 1.0 / double(n_global);
    if (loss_sigma) *loss_sigma = float(double(w->w_sigma) * acc[0] * invN);
    if (loss_u) *loss_u = float(double(w->w_u) * acc[1] * invN);
}

}  // extern "C"
