// Shared between the host API (tg_api.cu) and the per-group-size kernel translation units.
#ifndef TG_SHAPE_H
#define TG_SHAPE_H
#include <cuda_runtime.h>
#include <stddef.h>
#include "tg_spec.h"

struct TgShape {
    int sp[TG_SP_COUNT];
    TgLayout L;
};

// ---------------------------------------------------------------------------
// Shapes with kernel instantiations of their own.  The stage kernels are templates on FIX: 0 = the descriptor is a
// kernel argument (any shape); k > 0 = the descriptor is the compile-time constant below, so the whole TgLayout
// (sizes, row / parameter offsets, which constraint blocks exist) folds into the code: workspace arrays sit at
// constant offsets, absent constraint kinds are compiled out, loop bounds are known.  Same arithmetic in the same
// order, but the compiler contracts the folded code into FMAs differently in places: the objective and its gradient
// are bit-identical to the generic instantiation, constraint rows and their Jacobian may differ in the last places
// (C4: bit-identical throughout; tests/test_eval_sweep.py).  The list holds the BASELINE.json configurations
// (trajectory_generator_b200/synthetic.py builds the same descriptors; tests/test_packing.py compares them).
// ---------------------------------------------------------------------------
#define TG_FIXED_SHAPES 5
enum { TG_FIX_C2 = 1, TG_FIX_C3, TG_FIX_C4, TG_FIX_C5A, TG_FIX_C5C };
TG_HD constexpr int tg_fixed_spec(int fix, int field)
{
    constexpr int T[TG_FIXED_SHAPES][TG_SP_COUNT] = {
        // C2: 2-D, 8 control points, start / end velocity, v_max, a_max, angular-rate bound, 8 obstacles
        {2, 8, 5, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 2, 0, 0, 0, 0, 0, 0, 0, 0, 0, 8},
        // C3: 2-D, 17 control points, two intermediate waypoints with velocities, v_max, curvature bound
        {2, 17, 5, 0, 0, 0, 1, 0, 0, 1, 0, 2, 1, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0},
        // C4: 3-D, 11 control points, start velocity, zero-velocity end, v_max, a_max, 4 corridors x 2 intervals
        {3, 11, 2, 0, 1, 0, 1, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 4, 2, 2, 2, 2, 0, 0, 0, 0, 0},
        // C5a / C5c: 2-D, 8 control points, start / end velocity, v_max, a_max, angular-rate / curvature bound
        {2, 8, 5, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 2, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0},
        {2, 8, 5, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}};
    return T[fix - 1][field];
}

// index of the fixed shape equal to `sp`, 0 if none (host)
static inline int tg_fixed_index(const int *sp)
{
    for (int k = 1; k <= TG_FIXED_SHAPES; k++) {
        bool same = true;
        for (int i = 0; i < TG_SP_COUNT; i++) same = same && sp[i] == tg_fixed_spec(k, i);
        if (same) return k;
    }
    return 0;
}

#if defined(__CUDACC__)
// descriptor and layout a stage kernel works with: the kernel argument (FIX == 0) or compile-time constants
template <int FIX>
static __device__ __forceinline__ void tg_resolve_shape(const int *arg_sp, const TgLayout &arg_L, int *fsp, TgLayout *fL,
                                                        const int **sp, const TgLayout **L)
{
    if (FIX > 0) {
#pragma unroll
        for (int i = 0; i < TG_SP_COUNT; i++) fsp[i] = tg_fixed_spec(FIX > 0 ? FIX : 1, i);
        tg_make_layout(fsp, fL);
        *sp = fsp; *L = fL;
    } else {
        *sp = arg_sp; *L = &arg_L;
    }
}
#endif

// round bookkeeping of the lock-step solve (device memory).  Round r works through list[r & 1] (count[r & 1]
// problem indices, handed out through the head_* cursors) and the QP stage appends the problems that are not
// finished to the other list; `done` counts finished problems (polled by the host).
struct TgRoundCtl {
    int count[2], head_ls[2], head_qp[2], head_fd[2], done, pad;
    double flops_qp;      // sum over the chunk's problems of the QP stage's model flop count (written by the finish kernel)
};
#define TG_ROUNDCTL_BYTES 256

// Shapes whose per-problem scratch does not fit in shared memory run stage kernels that take it from the solve
// workspace instead: one slot per resident lane group (the grids are persistent, a group reuses its slot for every
// problem it pulls).  Their grids are capped at TG_FAR_CTAS_PER_SM CTAs per SM, so that the slot count is known before
// the launch (tg_plan_solve sizes the workspace); that is also their launch bound, which leaves them 256 registers a
// thread (no spills) and keeps the slots of a large shape few.  Only the generic instantiations exist: the QP kernel with 64 lanes
// (tg_solve_g64.cu), the line-search and derivative kernels with 32 (tg_solve_g32.cu, tg_solve_fd_g32.cu).
#define TG_FAR_CTAS_PER_SM 2

// Every kernel with dynamic shared memory is allowed the device's opt-in maximum (not the size of the launch at
// hand: launches of one kernel with different sizes may be issued from several host threads, tg_solve_mixed_host).
// Done once per (device, kernel).
#include <mutex>
#include <set>
#include <utility>
template <typename K>
static inline cudaError_t tg_allow_shared_memory(K kernel)
{
    static std::mutex mu;
    static std::set<std::pair<int, const void *>> done;
    int dev = 0, optin = 0;
    cudaError_t e;
    if ((e = cudaGetDevice(&dev))) return e;
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<int, const void *> key(dev, (const void *)kernel);
    if (done.count(key)) return cudaSuccess;
    cudaFuncAttributes attr;
    if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev))) return e;
    if ((e = cudaFuncGetAttributes(&attr, kernel))) return e;
    // static + dynamic <= the opt-in limit
    if ((e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)attr.sharedSizeBytes))) return e;
    done.insert(key);
    return cudaSuccess;
}

#define TG_DECLARE_VARIANT(SFX)                                                                                           \
    cudaError_t tg_launch_eval##SFX(const TgShape &S, int B, const double *par, const double *x, double *f, double *g,    \
                                    double *c, double *jnl, int sm_count, int smem_optin, cudaStream_t st);               \
    cudaError_t tg_launch_linear##SFX(const TgShape &S, int B, const double *par, double *alin, int sm_count,             \
                                      cudaStream_t st);                                                                   \
    size_t tg_eval_smem##SFX(const TgShape &S, bool sink_c, int smem_optin);                                              \
    cudaError_t tg_launch_begin##SFX(const TgShape &S, int B, const double *x, double *pws, size_t np, int maxiter,       \
                                     double ftol, int flags, TgRoundCtl *rc, int *list0, cudaStream_t st);                \
    cudaError_t tg_launch_ls##SFX(const TgShape &S, int B, const double *par, double *pws, size_t np, size_t smem,        \
                                  double *far, TgRoundCtl *rc, const int *list, int parity, int sm_count,                 \
                                  cudaStream_t st);                                                                       \
    cudaError_t tg_launch_qp##SFX(const TgShape &S, int B, double *pws, size_t np, int staged, size_t smem, double *far,  \
                                  TgRoundCtl *rc, const int *list, int *next, int parity, int sm_count, cudaStream_t st); \
    size_t tg_ls_smem##SFX(const TgShape &S);                                                                             \
    size_t tg_qp_smem##SFX(const TgShape &S, int staged);                                                                 \
    cudaError_t tg_launch_finish##SFX(const TgShape &S, int B, const double *pws, size_t np, double *x, double *f,        \
                                      int *status, int *nit, int *violation, TgRoundCtl *rc, cudaStream_t st);

TG_DECLARE_VARIANT(_g8)
TG_DECLARE_VARIANT(_g16)
TG_DECLARE_VARIANT(_g32)

// finite-difference stage (tg_solve_fd_g*.cu): value-only evaluators inlined, one kernel of its own
#define TG_DECLARE_FD(SFX)                                                                                              \
    cudaError_t tg_launch_fd##SFX(const TgShape &S, int B, const double *par, double *pws, size_t np, size_t smem,      \
                                  double *far, TgRoundCtl *rc, const int *list, int parity, int sm_count, cudaStream_t st);
TG_DECLARE_FD(_g8)
TG_DECLARE_FD(_g16)
TG_DECLARE_FD(_g32)

// QP stage with 64 lanes per problem (tg_solve_g64.cu)
cudaError_t tg_launch_qp_g64(const TgShape &S, int B, double *pws, size_t np, int staged, size_t smem, double *far,
                             TgRoundCtl *rc, const int *list, int *next, int parity, int sm_count, cudaStream_t st);
size_t tg_qp_smem_g64(const TgShape &S, int staged);

// launch counter of the library (tg_launch_count), for kernels launched outside tg_api.cu
void tg_note_launch(int count);

// fused kernel (group size 32 only)
cudaError_t tg_launch_fused_g32(const TgShape &S, int B, const double *par, double *x, double *f, int *status, int *nit,
                                int *violation, int maxiter, double ftol, int flags, double *gws, size_t ws_doubles,
                                int warps_per_cta, int ctas, size_t smem, int *queue, cudaStream_t st);
#endif
