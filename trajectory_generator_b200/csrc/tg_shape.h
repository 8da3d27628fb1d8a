// Shared between the host API (tg_api.cu) and the per-group-size kernel translation units: the shape a kernel is
// launched for, the fixed shapes with instantiations of their own, and the launchers with their arguments.
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

// Launchers of the device code (per lanes per problem: the tg_*_g<lanes>.cu translation units).  The host plan
// (tg_api.cu: tg_plan_solve, tg_eval_batch) decides every launch parameter; a launcher picks the instantiation for the
// fixed-shape index, the dimension and the placement it is handed and launches it.
//
// Lock-step stage kernels (tg_kernels_solve.inc).  tg_solve_phased fills one TgStageLaunch per slice and round and sets
// the stage's shared memory and workspace slots (far != nullptr: scratch in global memory) before each launch.
struct TgStageLaunch {
    TgShape S;
    int B;                  // problems of the slice (the grids are capped at the work)
    const double *par;      // parameter rows of the slice
    double *pws;            // persistent state of the slice's problems, np doubles each
    size_t np;
    size_t smem;            // dynamic shared memory of the stage's CTAs
    double *far;            // workspace slots of the stage, or nullptr
    int staged;             // QP stage: the persistent state is staged through shared memory
    TgRoundCtl *rc;
    const int *list;        // this round's list of unfinished problems
    int *next;              // QP stage: the next round's list
    int parity;             // round & 1
    int sm_count, fix;      // fix: tg_fixed_index of the shape, 0 = generic instantiations
    cudaStream_t st;
};
cudaError_t tg_launch_ls_g8(const TgStageLaunch &a), tg_launch_ls_g16(const TgStageLaunch &a), tg_launch_ls_g32(const TgStageLaunch &a);
cudaError_t tg_launch_fd_g8(const TgStageLaunch &a), tg_launch_fd_g16(const TgStageLaunch &a), tg_launch_fd_g32(const TgStageLaunch &a);
cudaError_t tg_launch_qp_g16(const TgStageLaunch &a), tg_launch_qp_g32(const TgStageLaunch &a), tg_launch_qp_g64(const TgStageLaunch &a);
// once per solve (32 lanes); the finish kernel writes lam[B*m] / kkt[B*4] (tg_sqp_kkt) unless they are null
cudaError_t tg_launch_begin_g32(const TgShape &S, int B, const double *x, double *pws, size_t np, int maxiter, double ftol,
                                int flags, TgRoundCtl *rc, int *list0, cudaStream_t st);
cudaError_t tg_launch_finish_g32(const TgShape &S, int B, const double *pws, size_t np, double *x, double *f, int *status,
                                 int *nit, int *violation, double *lam, double *kkt, TgRoundCtl *rc, cudaStream_t st);

// Evaluation kernel (tg_kernels_eval.inc): `groups` lane groups per CTA with `smem` bytes of shared memory
struct TgEvalLaunch {
    TgShape S;
    int B;
    const double *par, *x;
    double *f, *g, *c, *jnl;
    int fix, grid, groups;
    size_t smem;
    cudaStream_t st;
};
cudaError_t tg_launch_eval_g8(const TgEvalLaunch &a), tg_launch_eval_g16(const TgEvalLaunch &a), tg_launch_eval_g32(const TgEvalLaunch &a);
cudaError_t tg_launch_linear_g32(const TgShape &S, int B, const double *par, double *alin, int sm_count, cudaStream_t st);

// Multi-start selection kernel (tg_kernels_eval.inc, planned like the evaluation kernel by tg_multistart_select): one
// lane group per problem, its K starts' rows xs / f / status / nit / violation at b * K + k
struct TgSelectLaunch {
    TgShape S;
    int B, K;
    const double *par, *xs, *f;
    const int *status, *nit, *violation;
    double tol;
    double *x_best, *f_best;
    int *status_best, *nit_best, *violation_best, *best_start;
    double *max_violation;      // [B * K] or nullptr
    int fix, grid, groups;
    size_t smem;
    cudaStream_t st;
};
cudaError_t tg_launch_select_g8(const TgSelectLaunch &a), tg_launch_select_g16(const TgSelectLaunch &a),
    tg_launch_select_g32(const TgSelectLaunch &a);
// Post-solve polish kernel (tg_kernels_polish.inc, planned by tg_plan_polish): `groups` lane groups per CTA, each with
// tg_polish_group_doubles of scratch in `smem` (far == nullptr) or in its slot of `far`
struct TgPolishLaunch {
    TgShape S;
    int B;
    const double *par;
    double *x, *f;
    const int *status;
    int *violation;
    double *lam, *kkt;
    int *polish_status, *polish_iters;
    int maxiter;
    double tol;
    double *far;
    int fix, grid, groups;
    size_t smem;
    cudaStream_t st;
};
cudaError_t tg_launch_polish_g8(const TgPolishLaunch &a), tg_launch_polish_g16(const TgPolishLaunch &a),
    tg_launch_polish_g32(const TgPolishLaunch &a);
// Parameter-sensitivity kernel (tg_kernels_sens.inc, planned by tg_plan_polish with tg_sens_group_doubles of scratch);
// f_bar may be nullptr (zeros)
struct TgSensLaunch {
    TgShape S;
    int B;
    const double *par, *x;
    const int *status;
    const double *lam, *x_bar, *f_bar;
    double *par_bar;
    int *sens_status;
    double tol;
    double *far;
    int fix, grid, groups;
    size_t smem;
    cudaStream_t st;
};
cudaError_t tg_launch_sens_g8(const TgSensLaunch &a), tg_launch_sens_g16(const TgSensLaunch &a),
    tg_launch_sens_g32(const TgSensLaunch &a);
// Multi-start expansion (tg_multistart.cu)
cudaError_t tg_launch_multistart_expand(const TgLayout &L, int B, int K, const double *par, const double *x0,
                                        unsigned long long seed, double spread, double *par_out, double *x_out,
                                        int sm_count, cudaStream_t st);

// launch counter of the library (tg_launch_count), for kernels launched outside tg_api.cu
void tg_note_launch(int count);

// fused kernel (tg_solve_fused.cu, 32 lanes): it sizes its grid and its global workspace itself (the same numbers for both)
size_t tg_fused_workspace_bytes(const TgShape &S, int B, int sm_count, int smem_optin);
cudaError_t tg_launch_fused_g32(const TgShape &S, int B, const double *par, double *x, double *f, int *status, int *nit,
                                int *violation, double *lam, double *kkt, int maxiter, double ftol, int flags, void *gws,
                                int *queue, int sm_count, int smem_optin, cudaStream_t st);
#endif
