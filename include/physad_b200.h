/*
 * physad_b200.h -- C-ABI of the B200-native (sm_100a) phys-autodiff hot path.
 *
 * This is the drop-in boundary: plain C, POD structs, raw pointers and sizes, an int status on
 * every call (0 = ok; otherwise a cudaError_t value or PHYSAD_E_*), no torch / C++ types.  The
 * reference's C++ API (include/backend.h, mlp.h, mlp_grid.h, phys.h -- host-pointer, void-returning
 * free functions) is implemented in phys_autodiff_b200/csrc/cxx_api.cpp as thin wrappers over the
 * functions below; INTEGRATION.md shows the binding.  Each entry point cites the reference
 * interface it replaces (paths relative to the reference repo).
 *
 * Conventions
 *   *_dev  : every data pointer is a DEVICE pointer on the current device; `stream` is a
 *            cudaStream_t passed as void* (NULL = legacy default stream); the call only enqueues.
 *   *_host : every data pointer is a HOST pointer (pageable is fine, as in the reference, whose
 *            API is host-pointer only -- include/phys.h:66); the call stages through device
 *            scratch owned by the context, runs the same kernels and blocks until results are
 *            back in the caller's buffers.
 *   Layouts follow the reference: linear index (z*ny + y)*nx + x, x fastest (src/phys_cpu.cpp:17-19);
 *   vector fields are channel-major [ux(0..N-1), uy, uz] (include/phys.h:20-21); MLP outputs are
 *   AoS [sigma,ux,uy,uz] per point (include/mlp_grid.h:16).
 *   There is no CPU fallback anywhere behind this header: without a CUDA device every compute
 *   entry point returns an error.
 *   Threading: a context is NOT thread-safe -- serialise calls on it (use one context per host thread or
 *   per stream).  The reducing calls (fused_loss*, phys_loss*) share per-context reduction scratch, so two of
 *   them on the same context must be ordered on the device (same stream, or an event between streams).
 */
#ifndef PHYSAD_B200_H
#define PHYSAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHYSAD_ABI_VERSION 1

enum {
    PHYSAD_OK = 0,
    PHYSAD_E_INVALID = -1,     /* bad argument (null pointer, non-positive size, ...) */
    PHYSAD_E_UNSUPPORTED = -2, /* shape outside what the kernels are built for */
    PHYSAD_E_NOWEIGHTS = -3,   /* context has no weights yet */
    PHYSAD_E_PEER_TIMEOUT = -4 /* in-kernel multi-GPU exchange: a peer rank never arrived */
};

/* phys::GridSpec, include/phys.h:8-13 (bool widened to int for C). */
typedef struct physad_grid {
    int nx, ny, nz;
    float hx, hy, hz;
    float dt;
    int periodic;
} physad_grid;

/* phys::PhysWeights, include/phys.h:15-18. */
typedef struct physad_phys_weights {
    float w_sigma, w_u;
} physad_phys_weights;

/* phys::MLPDims + phys::CoordNorm, include/mlp_grid.h:13-17,26.  norm: 0 = ZeroToOne, 1 = MinusOneToOne. */
typedef struct physad_mlp_config {
    int In, H, Out;
    int norm;
} physad_mlp_config;

/* z-slab of the global grid owned by one rank: planes [z_begin, z_end).  Coordinates, wrap and
 * clamp always refer to the GLOBAL grid; halo planes are recomputed, never exchanged. */
typedef struct physad_slab {
    int z_begin, z_end;
} physad_slab;

typedef struct physad_ctx physad_ctx; /* opaque: resident weights, reduction scratch, staging */

int physad_abi_version(void);
/* Message for the last non-zero status returned on this thread ("" if none). */
const char* physad_last_error(void);
const char* physad_error_string(int status);

/* ---- context --------------------------------------------------------------------------- */
/* Binds to CUDA device `device` (-1 = current).  Fails if no sm_100 device is present. */
int physad_ctx_create(physad_ctx** out, int device);
int physad_ctx_destroy(physad_ctx* ctx);
/* Number of SMs of the bound device (grid sizing is derived from it). */
int physad_ctx_sm_count(const physad_ctx* ctx);

/* Make weights resident.  HOST pointers, layouts of phys::MLPWeights (include/mlp_grid.h:19-24):
 * W1[H*In] row-major, b1[H], W2[Out*H] row-major, b2[Out].  Replaces the per-call upload in
 * mlp_forward<ExecCuda> (src/mlp_cuda.cu:102-106).  Cheap (a few KB); call again after an update. */
int physad_set_weights(physad_ctx* ctx, const physad_mlp_config* cfg, const float* W1, const float* b1,
                       const float* W2, const float* b2);

/* ---- MLP operator ---------------------------------------------------------------------- */
/* y[B*Out] = MLP(x[B*In]) with the context's weights; any In/H/Out that fits shared memory.
 * Replaces mlp_forward<ExecCuda> (include/mlp.h:5-6, src/mlp_cuda.cu:91-121) / mlp_infer_cuda
 * (include/mlp_grid.h:41).  Bit-exact with mlp_forward<ExecCpu> (src/mlp_cpu.cpp:14-36). */
int physad_mlp_forward_dev(physad_ctx* ctx, const float* x, float* y, size_t B, void* stream);
int physad_mlp_forward_host(physad_ctx* ctx, const float* x, float* y, size_t B);

/* MSE weight gradients of the same MLP: dW1[H*In], db1[H], dW2[Out*H], db2[Out] for inputs x[B*In]
 * and targets y_target[B*Out], loss = mean((y - y_target)^2).  Replaces mlp_backward<ExecCuda>
 * (include/mlp.h:8-9, src/mlp_cuda.cu:123-184).  Bit-exact with mlp_backward<ExecCpu>
 * (src/mlp_cpu.cpp:38-85), which fixes the algorithm to a sequential fp32 walk over the batch per
 * gradient entry (SURVEY.md section 8f rank 1: outside the grid->loss path, not tuned). */
int physad_mlp_backward_dev(physad_ctx* ctx, const float* x, const float* y_target, float* dW1, float* db1, float* dW2,
                            float* db2, size_t B, void* stream);
int physad_mlp_backward_host(physad_ctx* ctx, const float* x, const float* y_target, float* dW1, float* db1,
                             float* dW2, float* db2, size_t B);

/* MLP over the grid at time t, coordinates generated from the point index (never materialised).
 * out: AoS [slab points][4].  Replaces mlp_grid_infer_cuda (include/mlp_grid.h:45,
 * src/mlp_grid.cpp:61-67).  Requires In = Out = 4. */
int physad_mlp_grid_infer_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float* out,
                              void* stream);
int physad_mlp_grid_infer_host(physad_ctx* ctx, const physad_grid* g, float t, float* out);

/* Six physics input fields at t-dt, t, t+dt in one pass (sigma_*: n, u_*: 3n channel-major, n =
 * slab points).  Replaces mlp_generate_fields_cuda (include/mlp_grid.h:55-57, src/mlp_grid.cpp:95-106). */
int physad_mlp_generate_fields_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float dt,
                                   float* sigma_tm1, float* sigma_t, float* sigma_tp1, float* u_tm1, float* u_t,
                                   float* u_tp1, void* stream);
int physad_mlp_generate_fields_host(physad_ctx* ctx, const physad_grid* g, float t, float dt, float* sigma_tm1,
                                    float* sigma_t, float* sigma_tp1, float* u_tm1, float* u_t, float* u_tp1);

/* ---- deeper MLPs (ADDITIVE: BASELINE config 5, depth sweep) ------------------------------------
 * 4 -> H -> H -> ... -> H -> 4 with `hidden_layers` >= 1 hidden layers of width H (H = 32, 64 or 128).  The
 * reference API has exactly one hidden layer (include/mlp.h:5-6); further layers repeat its layer rule
 * (src/mlp_cpu.cpp:19-24: from the bias, + W[g,h]*a[h] for h ascending, separate fp32 multiply and add,
 * ReLU).  There is no reference implementation for hidden_layers > 1 (parity is against oracle/oracle.c's
 * restatement only); hidden_layers == 1 is bit-identical to the one-hidden-layer entry points.
 * Wh: (hidden_layers-1) matrices [H x H] row-major [g][h]; bh: (hidden_layers-1) x H.  HOST pointers.
 * While the context holds a network of hidden_layers > 1, every entry point that evaluates the one-hidden-layer network
 * (physad_mlp_forward_*, physad_mlp_backward_*, physad_mlp_grid_infer_*, physad_mlp_generate_fields_*, physad_fused_loss_*,
 * physad_tangent_loss_*, physad_fused_loss_grad_*, physad_tangent_loss_grad_*) returns PHYSAD_E_UNSUPPORTED and writes
 * nothing; the host forms that take new weights (cfg != NULL) replace the network first and run.  Use the *_deep_* and
 * deep_* counterparts: physad_mlp_forward_deep_* for physad_mlp_forward_*, physad_deep_data_loss_grad_* for
 * physad_mlp_backward_*, physad_mlp_grid_infer_deep_dev, physad_mlp_generate_fields_deep_dev, physad_deep_loss_host,
 * physad_deep_loss_grad_*, physad_deep_tangent_loss_* and, at arbitrary points, physad_deep_tangent_points_loss_*.
 * hidden_layers == 1 is accepted everywhere.  A refused call leaves the previous network in place.
 * A later physad_set_weights() switches the context back to a one-hidden-layer network. */
int physad_set_weights_deep(physad_ctx* ctx, const physad_mlp_config* cfg, int hidden_layers, const float* W1,
                            const float* b1, const float* Wh, const float* bh, const float* W2, const float* b2);
/* How the hidden -> hidden layers of the deep entry points are evaluated (ADDITIVE; default 0).
 *   0: strict fp32 on the CUDA cores -- bit-identical to the CPU restatement (the parity mode);
 *   1: tcgen05 tensor cores, every fp32 operand split into three bf16 terms, six term products accumulated in fp32
 *      (deep_tc_kernels.cuh): NOT bit-exact -- outputs agree with mode 0 to ~1e-6 relative, the error class of an
 *      FFMA-contracted evaluation such as the reference's own CUDA kernels (src/mlp_cuda.cu).  Needs hidden_layers >= 2
 *      (with one hidden layer there is no hidden -> hidden contraction: PHYSAD_E_UNSUPPORTED from the forced deep kernel;
 *      the default route for one hidden layer is the reference-pinned kernel in either mode).  Layer images stay resident
 *      in shared memory when they fit (H = 128: <= 3 hidden layers), else they are streamed from L2; at H <= 64 two row
 *      tiles are in flight per SM.  Layer 1 stays strict. */
int physad_set_deep_mode(physad_ctx* ctx, int mode);
/* The operand image mode 1 keeps of ONE hidden -> hidden layer (host function, no GPU needed; physad_set_weights_deep calls
 * it): W = [H out][H in] row-major -> three bf16 terms t1 + t2 + t3 = W (each the round-to-nearest bf16 of what the previous
 * ones left), term p at element offset p*H*H, element (g, h) of a term at (h/8)*(H/8)*64 + (g/8)*64 + (g%8)*8 + (h%8): the
 * "K-major, no swizzle" core-matrix layout of a tcgen05 shared-memory descriptor with SBO = 128 B, LBO = 16*H B.
 * physad_deep_tc_layer_bytes(H) = 3*H*H*2 (0 for widths that are not built). */
size_t physad_deep_tc_layer_bytes(int H);
int physad_deep_tc_pack_layer(int H, const float* W, unsigned char* image);
/* Stage-wise evaluation over the grid (coordinates from the index); outputs as the one-layer calls above. */
int physad_mlp_grid_infer_deep_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float* out,
                                   void* stream);
int physad_mlp_generate_fields_deep_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float dt,
                                        float* sigma_tm1, float* sigma_t, float* sigma_tp1, float* u_tm1, float* u_t,
                                        float* u_tp1, void* stream);
/* One call for the depth sweep: the deep network's six fields (context scratch, 48 B per point) -> the residual loss of
 * src/phys_cpu.cpp:112-149 -> the two losses on the host.  Stage-wise inside (the MLP is 50-700x the stencil's time at these
 * depths, so fusing them would save < 3 %); the arithmetic follows physad_set_deep_mode. */
int physad_deep_loss_host(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, float t, float dt,
                          float* loss_sigma, float* loss_u);

/* ---- physics operators on supplied fields (whole grid, single device) -------------------- */
/* Residuals.  Replaces cuda_phys_residuals_fused / _nonfused (include/phys.h:67-77,120-130).
 * kernel_ms (host pointer, may be NULL) receives the kernel-only time of the _host variant, as the
 * reference's *_timed wrappers report (include/phys.h:106-117,145-156). */
int physad_phys_residuals_dev(physad_ctx* ctx, const physad_grid* g, const float* sigma_tm1, const float* sigma_t,
                              const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                              float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);
int physad_phys_residuals_host(physad_ctx* ctx, const physad_grid* g, const float* sigma_tm1, const float* sigma_t,
                               const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                               float* R_sigma, float* R_ux, float* R_uy, float* R_uz, float* kernel_ms);

/* Loss forward with the reduction ON THE DEVICE (the reference sums on the host,
 * src/phys_cuda_nonfused.cu:385-393).  acc_dev[2] (device, double) receives {sum R_sigma^2,
 * sum |R_u|^2}; R_* may be NULL.  Replaces cuda_phys_loss_forward_nonfused (include/phys.h:79-92)
 * and supplies the cuda_phys_loss_forward_fused the reference only planned
 * (docs/PLAN_FUSED_PHYS_LOSS.md:59). */
int physad_phys_loss_dev(physad_ctx* ctx, const physad_grid* g, const float* sigma_tm1, const float* sigma_t,
                         const float* sigma_tp1, const float* u_tm1, const float* u_t, const float* u_tp1,
                         double* acc_dev, float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);
int physad_phys_loss_host(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, const float* sigma_tm1,
                          const float* sigma_t, const float* sigma_tp1, const float* u_tm1, const float* u_t,
                          const float* u_tp1, float* loss_sigma, float* loss_u, float* R_sigma, float* R_ux,
                          float* R_uy, float* R_uz);

/* ---- reduced-precision field I/O (ADDITIVE: the reference plans it, REQUIREMENT.md:123-128 -- "inputs / outputs may be
 * FP16, differences and reductions keep FP32 accumulation" -- and never ships it) ------------------------------------
 * The six physics input fields live in HBM as 16-bit elements (dtype PHYSAD_F16 = IEEE half, PHYSAD_BF16 = bfloat16; same
 * layouts as above, element count unchanged): physad_mlp_generate_fields_lp_dev rounds the strict-fp32 MLP outputs to
 * nearest-even on the store, physad_phys_loss_lp_dev widens every load to fp32 and then runs the fp32 stencil, the double
 * reduction and (optionally) fp32 residual outputs unchanged: 24 instead of 48 B/point of input traffic.  Whole grid,
 * central scheme, nx % 4 == 0, 8-byte aligned field arrays.  What the rounding costs: with the reference's dt = 2e-3 the
 * time difference multiplies the rounding error of the fields by 1/(2 dt) = 250, see profiles/r02_lowprecision_io_study.json. */
enum { PHYSAD_F32 = 0, PHYSAD_F16 = 1, PHYSAD_BF16 = 2 };
int physad_mlp_generate_fields_lp_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float dt, int dtype,
                                      void* sigma_tm1, void* sigma_t, void* sigma_tp1, void* u_tm1, void* u_t, void* u_tp1,
                                      void* stream);
int physad_phys_loss_lp_dev(physad_ctx* ctx, const physad_grid* g, int dtype, const void* sigma_tm1, const void* sigma_t,
                            const void* sigma_tp1, const void* u_tm1, const void* u_t, const void* u_tp1, double* acc_dev,
                            float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);

/* The same on one rank's z-slab of supplied fields (multi-GPU, SURVEY.md section 8f rank 2): the six arrays
 * hold only the slab's planes (sigma_*: n, u_*: 3n channel-major, n = slab points); halo_lo / halo_hi
 * ([4 channels: sigma_t, ux_t, uy_t, uz_t][ny][nx] each, device) are the time-t planes just below / above the
 * slab in the GLOBAL grid with the wrap/clamp rule already applied -- the host obtains them from the
 * neighbouring ranks (ops.Context.phys_loss_sharded all-gathers the boundary planes with torch.distributed).
 * acc_dev[2] receives this slab's sums; R_* (slab-local) may be NULL. */
int physad_phys_loss_slab_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, const float* sigma_tm1,
                              const float* sigma_t, const float* sigma_tp1, const float* u_tm1, const float* u_t,
                              const float* u_tp1, const float* halo_lo, const float* halo_hi, double* acc_dev,
                              float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);

/* Residual VJP g = (2 w / float(N)) R.  Replaces cuda_phys_loss_backward_nonfused
 * (include/phys.h:94-103; CPU: src/phys_cpu.cpp:151-170). */
int physad_phys_backward_dev(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, const float* R_sigma,
                             const float* R_ux, const float* R_uy, const float* R_uz, float* g_sigma, float* g_ux,
                             float* g_uy, float* g_uz, void* stream);
int physad_phys_backward_host(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, const float* R_sigma,
                              const float* R_ux, const float* R_uy, const float* R_uz, float* g_sigma, float* g_ux,
                              float* g_uy, float* g_uz);
/* Same VJP recomputed from the fields.  Replaces cuda_phys_loss_backward_fused (include/phys.h:132-143). */
int physad_phys_backward_from_fields_dev(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w,
                                         const float* sigma_tm1, const float* sigma_t, const float* sigma_tp1,
                                         const float* u_tm1, const float* u_t, const float* u_tp1, float* g_sigma,
                                         float* g_ux, float* g_uy, float* g_uz, void* stream);
int physad_phys_backward_from_fields_host(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w,
                                          const float* sigma_tm1, const float* sigma_t, const float* sigma_tp1,
                                          const float* u_tm1, const float* u_t, const float* u_tp1, float* g_sigma,
                                          float* g_ux, float* g_uy, float* g_uz);

/* ---- the metric path: fused MLP + finite-difference residual + loss reduction ------------ */
/* One kernel: evaluates the MLP at (x,y,z,t-dt|t|t+dt) for every point of the slab (plus the
 * recomputed stencil halo), forms the residuals of src/phys_cpu.cpp:25-110 and reduces
 * {sum R_sigma^2, sum |R_u|^2} over the slab into acc_dev[2] (device, double).  No field ever
 * touches HBM.  R_* (device, slab-local, may be NULL) receive the residuals.  This composes
 * mlp_generate_fields_cuda + cuda_phys_loss_forward_* of the reference (call stack B/C of
 * SURVEY.md section 3); the reference has no such entry point (docs/BENCHMARK_REPORT.md:61).
 * Requires In = Out = 4.  After a multi-rank sum of acc_dev, physad_finalize_loss gives the loss. */
int physad_fused_loss_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float dt,
                          double* acc_dev, float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);
/* Host-buffer form: uploads the given weights, runs the kernel on the whole grid, returns the two
 * losses (and residuals if the pointers are non-NULL).  This is the call `e2e` in bench.py times. */
int physad_fused_loss_host(physad_ctx* ctx, const physad_grid* g, const physad_mlp_config* cfg, const float* W1,
                           const float* b1, const float* W2, const float* b2, const physad_phys_weights* w, float t,
                           float dt, float* loss_sigma, float* loss_u, float* R_sigma, float* R_ux, float* R_uy,
                           float* R_uz);
/* ---- multi-GPU: the same kernel with the all-reduce of the two sums done INSIDE it, over NVLink
 * peer memory (SURVEY.md section 8e asks for one collective of 2 doubles; this removes its launch).
 * Setup once per process group (one process per GPU, ranks of one node, world <= 8):
 *   1. every rank: physad_xchg_export(ctx, handle)            -> 64-byte CUDA IPC handle of its exchange buffer
 *   2. all-gather the handles with whatever the host uses (torch.distributed, MPI, a file ...)
 *   3. every rank: physad_xchg_connect(ctx, rank, world, handles)   -- handles: world x 64 bytes, in rank order
 * Then physad_fused_loss_allreduce_dev behaves like physad_fused_loss_dev, except that acc_dev
 * receives the GLOBAL sums on every rank (added in rank order: identical bits everywhere).  All ranks
 * must make the same sequence of these calls (one exchange epoch per call), slab empty or not.
 * CO-RESIDENCY: the exchanging kernels of all ranks wait for each other, so they must be able to run at the
 * same time -- one process per GPU, each rank launching on its own device (never two ranks' kernels queued
 * behind each other on one device or one stream).  A rank that never arrives makes the others give up after
 * ~4 s instead of hanging: their sums become NaN, physad_xchg_status() reports it, and the host one-call
 * form (physad_fused_loss_slab_host) returns PHYSAD_E_PEER_TIMEOUT. */
#define PHYSAD_XCHG_HANDLE_BYTES 64
int physad_xchg_export(physad_ctx* ctx, void* handle_out);
int physad_xchg_connect(physad_ctx* ctx, int rank, int world, const void* handles);
int physad_xchg_disconnect(physad_ctx* ctx);
int physad_fused_loss_allreduce_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, float dt,
                                    double* acc_dev, float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);
/* Synchronises the device, then *timed_out = 1 if any exchange since the last call gave up waiting for a peer
 * (and clears the flag), else 0. */
int physad_xchg_status(physad_ctx* ctx, int* timed_out);

/* One rank's whole step with host buffers in ONE call: (optionally) take new weights from the host,
 * run the fused kernel on `slab` (NULL = whole grid), whose last block stores the 16-byte result straight into
 * mapped pinned host memory (the host polls a sequence number: no copy, no stream synchronisation), and finalise.  exchange != 0 uses the in-kernel peer-memory all-reduce (after physad_xchg_connect), so
 * the returned losses are the GLOBAL ones on every rank; exchange == 0 returns this slab's share
 * (w * local sums / N_global).  This is the call bench.py's `e2e` times. */
int physad_fused_loss_slab_host(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab,
                                const physad_mlp_config* cfg, const float* W1, const float* b1, const float* W2,
                                const float* b2, const physad_phys_weights* w, float t, float dt, int exchange,
                                float* loss_sigma, float* loss_u);

/* L = float(w * acc * (1.0 / N_global)) exactly as src/phys_cpu.cpp:146-148.  Pure host arithmetic. */
void physad_finalize_loss(const double acc[2], const physad_phys_weights* w, size_t n_global, float* loss_sigma,
                          float* loss_u);

/* Weight initialiser of the grid driver for non-C++ hosts: uniform [-scale, scale] from
 * std::mt19937(seed) in the order W1, b1, W2, b2.  Replaces phys::mlp_random_init
 * (include/mlp_grid.h:34, src/mlp_grid.cpp:8-19).  HOST pointers; no device work. */
void physad_mlp_random_init(int In, int H, int Out, unsigned int seed, float scale, float* W1, float* b1, float* W2,
                            float* b2);

/* ---- analytic ("tangent") loss (ADDITIVE, explicitly NOT the parity path) --------------------------------------------
 * BASELINE.json's north_star in its literal wording: the input-derivatives are PROPAGATED THROUGH the MLP (forward mode,
 * dy/dx, dy/dy, dy/dz, dy/dt per point in registers) and the PDE residuals of src/phys_cpu.cpp:103-106 are formed from them
 * -- no finite differences, no second and third network evaluation, no halo.  The reference never does this (every
 * derivative there is a central difference of outputs sampled on the grid, SURVEY.md section 0 fact 1), so the result
 * differs from physad_fused_loss_dev by the discretisation error; the checker is oracle.c: oracle_tangent_loss (unpinned).
 * Space derivatives are with respect to the physical coordinate x = i*hx of the normalised network input.  acc_dev[2]
 * receives {sum R_sigma^2, sum |R_u|^2} over the slab (finalise with physad_finalize_loss after a multi-rank sum);
 * R_* (device, slab-local) optional.  Requires In = Out = 4, H <= 128. */
int physad_tangent_loss_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, double* acc_dev,
                            float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);
/* Host-buffer form on the whole grid: (optionally) new weights in, the two losses out. */
int physad_tangent_loss_host(physad_ctx* ctx, const physad_grid* g, const physad_mlp_config* cfg, const float* W1, const float* b1,
                             const float* W2, const float* b2, const physad_phys_weights* w, float t, float* loss_sigma,
                             float* loss_u);

/* ---- closed loop (ADDITIVE: the reference plans it, REQUIREMENT.md:155-169, but stops at dL/dR,
 * src/phys_cpu.cpp:151-170, and its MLP backward is the MSE one, src/mlp_cpu.cpp:38-85) ----------------
 * Loss of the MLP-generated fields AND the gradient of L_sigma + L_u (weights w included, mean over N) with
 * respect to the MLP weights set by physad_set_weights: forward stage-wise on the device (fields of the three
 * slices, residuals and the stencil adjoint kept in a context-owned workspace of 80 B/point), then two backward
 * kernels: the transposed stencil, and the back-propagation through the MLP with the weight-gradient reduction.  acc: 2 device doubles (sum R_sigma^2, sum |R_u|^2,
 * see physad_finalize_loss); grad: 9H+4 device doubles laid out  dW1[H*4] | db1[H] | dW2[4*H] | db2[4]  (the
 * reference's W1/b1/W2/b2 layouts).  Whole grid on one GPU.  The host form takes/returns host buffers (any
 * gradient pointer may be null) and replaces the weights first when cfg != NULL. */
int physad_fused_loss_grad_dev(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, float t, float dt,
                               double* acc, double* grad, void* stream);
/* One rank's share for multi-GPU: the SUMS over the points of slab [z_begin, z_end) -- acc as above and the partial
 * gradient (already scaled by 2w/N of the GLOBAL grid) -- so that an all-reduce(sum) of the 9H+6 doubles over the
 * ranks gives the whole-grid result.  The two residual planes and four field planes around the slab are recomputed
 * locally from coordinates (no halo exchange).  Empty slab: zeros. */
int physad_fused_loss_grad_slab_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab,
                                    const physad_phys_weights* w, float t, float dt, double* acc, double* grad, void* stream);
int physad_fused_loss_grad_host(physad_ctx* ctx, const physad_grid* g, const physad_mlp_config* cfg, const float* W1,
                                const float* b1, const float* W2, const float* b2, const physad_phys_weights* w, float t,
                                float dt, float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dW2, float* db2);

/* ---- closed loop of the analytic loss (ADDITIVE, no reference counterpart) ---------------------------------------------
 * physad_tangent_loss_dev's sums AND the gradient of L_sigma + L_u (weights w included, mean over the GLOBAL N) with
 * respect to the weights set by physad_set_weights: reverse mode over the forward-mode tangents, one persistent kernel
 * per call (points are independent: no stencil adjoint, no halo, no per-point workspace).  The forward arithmetic is
 * physad_tangent_loss_dev's, so acc equals its sums.  acc: 2 device doubles (sum R_sigma^2, sum |R_u|^2 over the slab);
 * grad: 9H+4 device doubles  dW1[H*4] | db1[H] | dW2[4*H] | db2[4]  (the reference's layouts), the slab's share already
 * scaled by 2w/N of the whole grid -- so an all-reduce(sum) of the 9H+6 doubles over the ranks' slabs gives the
 * whole-grid result.  slab NULL = whole grid; an empty slab gives zeros.  Requires In = Out = 4, H <= 128 and a
 * one-hidden-layer network (see physad_set_weights_deep).  Bitwise repeatable. */
int physad_tangent_loss_grad_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, const physad_phys_weights* w,
                                 float t, double* acc, double* grad, void* stream);
/* Host-buffer form on the whole grid: (optionally) new weights in, the two losses and the gradient out (any output
 * pointer may be null). */
int physad_tangent_loss_grad_host(physad_ctx* ctx, const physad_grid* g, const physad_mlp_config* cfg, const float* W1,
                                  const float* b1, const float* W2, const float* b2, const physad_phys_weights* w, float t,
                                  float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dW2, float* db2);

/* ---- closed loop of deeper networks (ADDITIVE, no reference counterpart) -------------------------------------------------
 * The finite-difference loss of physad_deep_loss_host AND the gradient of L_sigma + L_u (weights w included, mean over the
 * GLOBAL N) with respect to every layer of the network set by physad_set_weights_deep (strict fp32 arithmetic, mode 0).
 * Forward stage-wise on the device (the deep fields of the three slices, residuals and the stencil adjoint in the
 * context's workspace of 80 B/point), then one persistent kernel that recomputes the hidden layers tile by tile in the
 * forward's exact order (so the ReLU masks are those of the fields that produced R), keeps each layer's activations in a
 * per-block checkpoint area (L x 96 KB per SM) and back-propagates through every layer, and a reduction of the block
 * partials in block order (bitwise repeatable).
 * acc: 2 device doubles (sum R_sigma^2, sum |R_u|^2 over the slab); grad: P = physad_deep_grad_len(H, L) device doubles
 *   dW1[H*4] | db1[H] | dWh[(L-1)*H*H, row-major [out][in]] | dbh[(L-1)*H] | dW2[4*H] | db2[4]
 * (the argument order of physad_set_weights_deep), the slab's share already scaled by 2w/N of the whole grid -- so an
 * all-reduce(sum) of the P+2 doubles over the ranks' slabs gives the whole-grid result.  slab NULL = whole grid; an empty
 * slab gives zeros; a slab recomputes the field planes two around it locally (no halo exchange).  L = 1 is the
 * one-hidden-layer closed loop (physad_fused_loss_grad_dev / _slab_dev), bit for bit.
 * Errors: no deep weights (or a physad_set_weights after them): PHYSAD_E_NOWEIGHTS; physad_set_deep_mode(1) or upwind
 * advection: PHYSAD_E_UNSUPPORTED; bad slab or null pointer: PHYSAD_E_INVALID; a recomputed window of 2^31 points or
 * more: PHYSAD_E_UNSUPPORTED.
 * physad_deep_grad_len: host-only, P(H, L) = 9H + 4 + (L-1)(H^2 + H), 0 for shapes that are not built. */
size_t physad_deep_grad_len(int H, int hidden_layers);
int physad_deep_loss_grad_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, const physad_phys_weights* w,
                              float t, float dt, double* acc, double* grad, void* stream);
/* Host-buffer form on the whole grid with the context's deep weights: the two losses and the gradient out, split into the
 * six arrays of physad_set_weights_deep's layouts (any output pointer may be null). */
int physad_deep_loss_grad_host(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, float t, float dt,
                               float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dWh, float* dbh, float* dW2,
                               float* db2);

/* ---- analytic loss of deeper networks and its closed loop (ADDITIVE, no reference counterpart) ---------------------------
 * The analytic loss of physad_tangent_loss_dev for the network set by physad_set_weights_deep: per point the network runs
 * on the value row and the four tangent rows d/dc_k (k = x, y, z, t), the value row in the strict fp32 order of
 * physad_mlp_grid_infer_deep (so the ReLU masks are that network's at time t), the tangent rows with fused multiply-adds
 * (inputs ascending); residuals and sums as physad_tangent_loss_dev.  One persistent kernel plus a block-order reduction
 * (bitwise repeatable); points are independent, so a slab needs no window and no halo.
 * physad_deep_tangent_loss_dev: acc = 2 device doubles (sum R_sigma^2, sum |R_u|^2 over the slab); R_* (all set or all
 *   null): slab-local residuals.
 * physad_deep_tangent_loss_grad_dev: the same acc (bit for bit) AND the gradient of L_sigma + L_u (weights w included,
 *   mean over the GLOBAL N) with respect to every layer, P = physad_deep_grad_len(H, L) device doubles in the layout of
 *   physad_deep_loss_grad_dev, the slab's share already scaled by 2w/N of the whole grid -- so an all-reduce(sum) of the
 *   P+2 doubles over the ranks' slabs gives the whole-grid result.  Reverse mode over the forward, in the same kernel:
 *   per-block activation checkpoints (L x 80 KB per SM), no per-point workspace.
 * slab NULL = whole grid; an empty slab gives zeros.  L = 1 is physad_tangent_loss_dev / physad_tangent_loss_grad_dev,
 * bit for bit.  The advection switch does not apply.
 * Errors: no deep weights (or a physad_set_weights after them): PHYSAD_E_NOWEIGHTS; physad_set_deep_mode(1):
 * PHYSAD_E_UNSUPPORTED; bad slab, null pointer or residual pointers not all set or all null: PHYSAD_E_INVALID; a grid of
 * 2^31 points or more (hence any such slab): PHYSAD_E_UNSUPPORTED. */
int physad_deep_tangent_loss_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, float t, double* acc,
                                 float* R_sigma, float* R_ux, float* R_uy, float* R_uz, void* stream);
int physad_deep_tangent_loss_grad_dev(physad_ctx* ctx, const physad_grid* g, const physad_slab* slab, const physad_phys_weights* w,
                                      float t, double* acc, double* grad, void* stream);
/* Host-buffer form on the whole grid with the context's deep weights: the two losses and the gradient out, split into the
 * six arrays of physad_set_weights_deep's layouts (any output pointer may be null). */
int physad_deep_tangent_loss_grad_host(physad_ctx* ctx, const physad_grid* g, const physad_phys_weights* w, float t,
                                       float* loss_sigma, float* loss_u, float* dW1, float* db1, float* dWh, float* dbh,
                                       float* dW2, float* db2);

/* ---- deeper networks at arbitrary points (ADDITIVE, no reference counterpart) ----------------------------------------
 * The network set by physad_set_weights_deep (any hidden_layers >= 1) evaluated at caller-supplied inputs, and a data-fit
 * loss with its gradient with respect to every layer: the term that anchors a physics-informed fit to initial conditions,
 * boundary values or observations (the physics residual alone is zero for every constant field).  Strict fp32 on the CUDA
 * cores (deep mode 0).
 * physad_mlp_forward_deep_*: y[B][4] = MLP(x[B][4]), x = the network's inputs (x, y, z, t) already normalised, like
 *   physad_mlp_forward's x.  The arithmetic of physad_mlp_grid_infer_deep (layer 1 from b1, + W1[h,k] x_k for k ascending,
 *   each product rounded; hidden and output layers from the bias, h ascending), so the outputs equal the CPU restatement
 *   oracle_mlp_forward_deep bit for bit, equal physad_mlp_grid_infer_deep's at the grid's own coordinates, and at
 *   hidden_layers == 1 equal physad_mlp_forward_*'s.  _dev: x and y DEVICE pointers, 16-byte aligned; no limit on B.
 * physad_deep_data_loss_grad_dev: L_d = (1/n_norm) sum_i sum_o lam[o] (y_io - target_io)^2 with y = MLP(x).
 *   lam: 4 HOST floats (finite, >= 0), or NULL for 1/4 each -- the mean((y - target)^2) of physad_mlp_backward.
 *   acc: 1 device double, the un-normalised weighted sum sum_i sum_o lam[o] (y_io - target_io)^2.
 *   grad: P = physad_deep_grad_len(H, L) device doubles in the layout of physad_deep_loss_grad_dev
 *   (dW1 | db1 | dWh | dbh | dW2 | db2), already scaled by 2 lam[o] / n_norm: with n_norm = the points of ALL shards, the
 *   shards' acc and grad add up (all-reduce(sum)), and grad adds directly to the physics gradient.  x, target: [B][4] device,
 *   16-byte aligned.  B = 0 (an empty shard) writes acc = 0 and a zero gradient.  Bitwise repeatable.
 * physad_deep_data_loss_grad_host: host arrays, n_norm = B; loss = L_d as float, the gradient split into the six arrays
 *   of physad_set_weights_deep's layouts (any output pointer may be null); B = 0 gives zeros.
 * Errors: no deep weights (or a physad_set_weights after them): PHYSAD_E_NOWEIGHTS; physad_set_deep_mode(1):
 * PHYSAD_E_UNSUPPORTED; n_norm == 0, a negative or non-finite lam, a null or misaligned pointer with B > 0 (acc and grad
 * always): PHYSAD_E_INVALID.  A refused call writes nothing. */
int physad_mlp_forward_deep_dev(physad_ctx* ctx, const float* x, float* y, size_t B, void* stream);
int physad_mlp_forward_deep_host(physad_ctx* ctx, const float* x, float* y, size_t B);
int physad_deep_data_loss_grad_dev(physad_ctx* ctx, const float* x, const float* target, size_t B, const float* lam,
                                   size_t n_norm, double* acc, double* grad, void* stream);
int physad_deep_data_loss_grad_host(physad_ctx* ctx, const float* x, const float* target, size_t B, const float* lam,
                                    float* loss, float* dW1, float* db1, float* dWh, float* dbh, float* dW2, float* db2);

/* ---- analytic loss of deeper networks at arbitrary points (ADDITIVE, no reference counterpart) ---------------------------
 * The physics loss of physad_deep_tangent_loss_* at caller-supplied collocation points (x, y, z, t) spread over the whole
 * space-time domain instead of the grid's points at one time: the term that makes a fit learn the dynamics between the
 * times where data anchor it.  The same kernel body as physad_deep_tangent_loss_* (strict fp32 value row, FMA tangent
 * rows, residuals, seeds and reverse mode), with one float4 load per point for the inputs and W1[h,3] t rounded per point;
 * so with x = the grid's points (in linear order) and dcdx = physad_grid_input_scales, the sums, residuals and gradient
 * equal the grid calls' bit for bit.  Any hidden_layers >= 1 (one hidden layer runs the same kernel).
 * physad_grid_input_scales: dc/dx of the three space inputs exactly as the grid's analytic calls form them
 *   (f / ((n-1) h), f = 2 for MinusOneToOne (norm 1), 1 for ZeroToOne (norm 0), 0 for an extent of 1).  Host-only, no GPU.
 * x: [B][4] DEVICE floats, 16-byte aligned: the network inputs, already normalised; the fourth is the grid calls' time input
 *   (t for MinusOneToOne, t + 0.5 for ZeroToOne), and d/dt is taken with respect to it (factor 1).
 * dcdx: 3 finite HOST floats, dc/dx of the three space inputs (the residual's d/dx_j = dcdx[j] d/dc_j).
 * physad_deep_tangent_points_loss_dev: acc = 2 device doubles (sum R_sigma^2, sum |R_u|^2 over the B points, not
 *   normalised); R: null or [B][4] device floats, 16-byte aligned, {R_sigma, R_ux, R_uy, R_uz} per point.
 * physad_deep_tangent_points_loss_grad_dev: the same acc (bit for bit) AND the gradient of L_sigma + L_u with
 *   L = (w / n_norm) sum R^2, P = physad_deep_grad_len(H, L) device doubles in the layout of physad_deep_loss_grad_dev,
 *   scaled by 2.f * w / float(n_norm): with n_norm = the points of ALL shards, the shards' P+2 doubles add up under one
 *   all-reduce(sum), and grad adds directly to physad_deep_data_loss_grad_dev's and to the grid calls' gradients.
 * physad_deep_tangent_points_loss_grad_host: x a host array, n_norm = B; the losses (physad_finalize_loss(acc, w, B)) and the
 *   gradient split into the six arrays of physad_set_weights_deep's layouts (any output pointer may be null).
 * B = 0 (an empty shard) writes zero sums and a zero gradient.  Bitwise repeatable.
 * Errors: no deep weights (or a physad_set_weights after them): PHYSAD_E_NOWEIGHTS; physad_set_deep_mode(1):
 * PHYSAD_E_UNSUPPORTED; a null pointer (x only with B > 0), a misaligned x or R (16 bytes) or acc or grad (8 bytes), a
 * non-finite dcdx, n_norm == 0, or (physad_grid_input_scales) a non-positive extent or a norm other than 0 or 1:
 * PHYSAD_E_INVALID.  A refused call writes nothing. */
int physad_grid_input_scales(const physad_grid* g, int norm, float dcdx[3]);
int physad_deep_tangent_points_loss_dev(physad_ctx* ctx, const float* x, size_t B, const float* dcdx, double* acc,
                                        float* R, void* stream);
int physad_deep_tangent_points_loss_grad_dev(physad_ctx* ctx, const float* x, size_t B, const float* dcdx,
                                             const physad_phys_weights* w, size_t n_norm, double* acc, double* grad,
                                             void* stream);
int physad_deep_tangent_points_loss_grad_host(physad_ctx* ctx, const float* x, size_t B, const float* dcdx,
                                              const physad_phys_weights* w, float* loss_sigma, float* loss_u, float* dW1,
                                              float* db1, float* dWh, float* dbh, float* dW2, float* db2);

/* Host-only: the work partition the fused kernel is launched with.  The sequence of tiles x planes
 * tile-planes (tile-major) is cut into at most `slots` contiguous ranges of equal cost, a range paying
 * ~0.9 plane-equivalents for every z-segment it starts (its recomputed halo planes).  Writes the
 * range boundaries (first = 0, last = tiles*planes) to out and returns their count (blocks + 1), or a
 * negative status.  Exposed so the partition can be tested without a GPU. */
int physad_plan_ranges(int tiles, int planes, int slots, int* out, int out_cap);

/* Residual arithmetic mode.  0 (default): the stencil and the residual sums in fp32 with fused multiply-adds,
 * like the reference's own CUDA kernels (measured within ~1e-7 * max|R| of the CPU reference; gate 1e-5).
 * 1: evaluated in double exactly as cpu_phys_residuals does (src/phys_cpu.cpp:66-109), so residuals are
 * BIT-IDENTICAL to the CPU reference (given the bit-exact MLP); costs ~5 % on the fused kernel and makes the
 * HBM-bound stage-wise kernels FP64/conversion-bound (0.24 -> 0.30 ms at 256^3).  Applies to the fused kernel
 * and to the stage-wise physics kernels.  Returns the previous value. */
int physad_set_exact_residuals(physad_ctx* ctx, int on);

/* Diagnostics: per-block timeline of the following fused launches.  dev_buf (DEVICE memory, zeroed by the caller)
 * holds blocks_cap x 18 x 2 uint64 {globaltimer ns, SM clock}: slot 0 block start, 1 prologue done, 2+3s / 3+3s /
 * 4+3s = z-segment s (< 4) start / first halo plane done / end, 14 march done, 15 {SM id, tile-planes owned},
 * 16 block exit.  NULL switches it off (default).  Used by tools/trace_fused.py. */
int physad_set_fused_trace(physad_ctx* ctx, unsigned long long* dev_buf, int blocks_cap);
/* Advection scheme of the STAGE-WISE physics operators (phys_residuals / phys_loss / phys_backward_from_fields, *_dev
 * and *_host).  0 (default): central differences, the reference (src/phys_cpu.cpp:80-93).  1: first-order UPWIND for the
 * advective derivatives of u . grad(f) -- (f - f_minus)/h where u_j > 0, (f_plus - f)/h otherwise; divergence and time
 * derivative stay central.  ADDITIVE: the reference plans this switch (REQUIREMENT.md:123-134: "consistent with the central
 * scheme for small velocities, no NaN on large random velocity fields") and never ships it, so parity is against
 * oracle/oracle.c's restatement only ("unpinned").  The fused kernel and the closed-loop gradient implement the central
 * scheme only and return PHYSAD_E_UNSUPPORTED while upwind is selected.  Returns the previous value (-1: bad argument). */
int physad_set_advection(physad_ctx* ctx, int scheme);
/* Tuning knob for experiments: selects the fused-kernel variant (0 = default). Returns the previous value. */
int physad_set_fused_variant(physad_ctx* ctx, int variant);
/* Number of kernel launches this context has enqueued since creation (bench.py's gpu_launches). */
uint64_t physad_launch_count(const physad_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* PHYSAD_B200_H */
