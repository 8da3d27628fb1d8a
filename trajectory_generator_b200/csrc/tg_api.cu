// Host side of the C-ABI declared in include/trajectory_generator_b200.h, plus the single-problem kernels
// behind the reference's 24 legacy symbols.
//
// Device code lives in per-group-size translation units (a problem is worked on by 8, 16, 32 or 64 lanes):
//   tg_eval_g*.cu      M1: objective, gradient, constraint rows, analytic nonlinear Jacobian rows
//   tg_solve_g*.cu     M2: the SLSQP iteration (tg_sqp.h) as lock-step stage kernels: line search, QP stage
//   tg_solve_fd_g*.cu  M2: the derivative stage
//   tg_solve_fused.cu  M2 as one kernel (kept for comparison)
// The plans here (tg_plan_solve, tg_eval_batch) make every launch decision -- lanes, shared memory, placement,
// staging, slices, fixed-shape instantiation -- and read the tuning overrides; the units' launchers execute them.
// Data layout in HBM: row-major [B][n] variables, [B][P] parameters, [B][m] rows, [B][m_nl][n] Jacobians --
// a lane group reads/writes its problem's rows as contiguous 8-byte accesses; per-problem working sets are
// staged in shared memory.
#include <assert.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <initializer_list>
#include <mutex>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "tg_sqp.h"
#include "tg_sens.h"
#include "tg_shape.h"
#include "../../include/trajectory_generator_b200.h"

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

static int tg_fail(int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (e != cudaSuccess) snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(g_err, sizeof g_err, "%s", what);
    return code;
}

#define TG_CUDA(call)                                                          \
    do {                                                                       \
        cudaError_t e_ = (call);                                               \
        if (e_ != cudaSuccess) return tg_fail(100 + (int)e_, #call, e_);       \
    } while (0)

static int tg_make_shape(const int *spec, TgShape *S)
{
    if (!spec) return tg_fail(1, "spec is NULL");
    memcpy(S->sp, spec, sizeof S->sp);
    const int d = spec[TG_SP_DIM], N = spec[TG_SP_NCP];
    if (d != 2 && d != 3) return tg_fail(2, "dimension must be 2 or 3");
    if (N < 4 || N > 512) return tg_fail(2, "number of control points out of range");
    if (spec[TG_SP_NCORR] < 0 || spec[TG_SP_NCORR] > TG_MAX_CORRIDORS) return tg_fail(2, "too many corridors");
    tg_make_layout(S->sp, &S->L);
    return 0;
}

// Everything that lives on a device (properties, cached staging buffers, streams) is kept per device id: a
// process may switch devices between calls (cudaSetDevice) and must never be handed another device's pointers.
#define TG_MAX_DEVICES 64
static thread_local int g_sm_count = 0, g_smem_optin = 0;      // of the calling thread's current device (tg_device_check)
static int g_dev_sm[TG_MAX_DEVICES], g_dev_smem[TG_MAX_DEVICES];
static std::atomic<int> g_dev_known[TG_MAX_DEVICES];
template <int D>
__global__ void tg_legacy_kernel(int what, const double *pts, int N, double alpha, int kind, const double *centers,
                                 const double *radii, int K, double *out);

extern "C" int tg_device_check(void)
{
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return tg_fail(10, "no CUDA device available (this library has no CPU path)", e);
    int dev = 0;
    TG_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= TG_MAX_DEVICES) return tg_fail(10, "device index out of range");
    if (!g_dev_known[dev].load(std::memory_order_acquire)) {
        cudaFuncAttributes attr;
        e = cudaFuncGetAttributes(&attr, tg_legacy_kernel<2>);
        if (e != cudaSuccess) return tg_fail(11, "no kernel image for this device (built for sm_100a)", e);
        int sm = 0, smem = 0;
        TG_CUDA(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev));
        TG_CUDA(cudaDeviceGetAttribute(&smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        g_dev_sm[dev] = sm; g_dev_smem[dev] = smem;
        g_dev_known[dev].store(1, std::memory_order_release);
    }
    g_sm_count = g_dev_sm[dev];
    g_smem_optin = g_dev_smem[dev];
    return 0;
}

extern "C" int tg_spec_count(void) { return TG_SP_COUNT; }

extern "C" int tg_layout(const int *spec, int *out, int cap)
{
    const int cnt = (int)(sizeof(TgLayout) / sizeof(int));
    if (spec && out && cap >= cnt) {
        TgLayout L;
        tg_make_layout(spec, &L);
        memcpy(out, &L, sizeof L);
    }
    return cnt;
}

extern "C" int tg_fixed_shape_index(const int *spec) { return spec ? tg_fixed_index(spec) : 0; }

extern "C" const char *tg_last_error(void) { return g_err; }
extern "C" unsigned long long tg_launch_count(void) { return g_launches.load(); }
void tg_note_launch(int count) { g_launches += (unsigned long long)count; }

// ---------------------------------------------------------------------------
// lanes per problem.  Heuristic: enough lanes for the per-interval terms (the longest per-lane chains), capped by
// what shared memory allows; TG_EVAL_GS / TG_LS_GS (8, 16, 32) and TG_QP_GS (16, 32, 64) override for tuning.
// ---------------------------------------------------------------------------
static int tg_env_gs(const char *name, int dflt)
{
    const char *v = getenv(name);
    if (!v) return dflt;
    const int g = atoi(v);
    return (g == 8 || g == 16 || g == 32) ? g : dflt;
}

static int tg_default_gs(const TgLayout &L)
{
    return L.nint <= 8 ? 8 : (L.nint <= 16 ? 16 : 32);
}

// launchers of a kernel family by lanes per problem (8, 16, 32, 64); nullptr: no such kernel, never planned
static int tg_lanes_index(int lanes) { return lanes == 8 ? 0 : lanes == 16 ? 1 : lanes == 32 ? 2 : 3; }
typedef cudaError_t (*TgStageLauncher)(const TgStageLaunch &);
static const TgStageLauncher tg_ls_launchers[4] = {tg_launch_ls_g8, tg_launch_ls_g16, tg_launch_ls_g32, nullptr};
static const TgStageLauncher tg_fd_launchers[4] = {tg_launch_fd_g8, tg_launch_fd_g16, tg_launch_fd_g32, nullptr};
static const TgStageLauncher tg_qp_launchers[4] = {nullptr, tg_launch_qp_g16, tg_launch_qp_g32, tg_launch_qp_g64};
static cudaError_t (*const tg_eval_launchers[3])(const TgEvalLaunch &) = {tg_launch_eval_g8, tg_launch_eval_g16, tg_launch_eval_g32};

// fixed-shape instantiation of a shape (tg_shape.h); TG_GENERIC_KERNELS: the generic ones, for A/B runs
static int tg_plan_fix(const TgShape &S) { return getenv("TG_GENERIC_KERNELS") ? 0 : tg_fixed_index(S.sp); }

extern "C" int tg_eval_batch(const int *spec, int B, const double *par, const double *x, double *f, double *g,
                             double *c, double *jnl, void *stream)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if ((rc = tg_device_check())) return rc;
    const int gs = tg_env_gs("TG_EVAL_GS", tg_default_gs(S.L));
    // (a CTA runs fewer lane groups where 128 / gs do not fit; one must)
    const int groups = tg_eval_groups(S.L, gs, c == nullptr, g_smem_optin);
    const size_t need = (size_t)tg_eval_group_doubles(S.L, c == nullptr) * sizeof(double);
    if (groups == 0) {
        snprintf(g_err, sizeof g_err, "tg_eval_kernel: a problem with n = %d, m = %d needs %zu bytes of shared memory, "
                 "more than the device's %d", S.L.n, S.L.m, need, g_smem_optin);
        return 3;
    }
    int grid = (B + groups - 1) / groups;
    if (grid > g_sm_count * 32) grid = g_sm_count * 32;
    const TgEvalLaunch a = {S, B, par, x, f, g, c, jnl, tg_plan_fix(S), grid, groups, groups * need, (cudaStream_t)stream};
    cudaError_t e = tg_eval_launchers[tg_lanes_index(gs)](a);
    g_launches++;
    if (e != cudaSuccess) return tg_fail(100 + (int)e, "tg_eval_kernel launch", e);
    return 0;
}

extern "C" int tg_linear_rows_batch(const int *spec, int B, const double *par, double *alin, void *stream)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if ((rc = tg_device_check())) return rc;
    cudaError_t e = tg_launch_linear_g32(S, B, par, alin, g_sm_count, (cudaStream_t)stream);
    g_launches++;
    if (e != cudaSuccess) return tg_fail(100 + (int)e, "tg_linear_kernel launch", e);
    return 0;
}

// ---------------------------------------------------------------------------
// M2 launch plan of the lock-step solve: every launch decision of tg_solve_phased, and the workspace it carves
// ---------------------------------------------------------------------------
#define TG_MAX_SLICES 4
struct TgStagePlan {
    int lanes, far;         // far: scratch in workspace slots instead of shared memory
    size_t smem;            // dynamic shared memory per CTA
};
struct TgSolvePlan {
    int fix;                // fixed-shape instantiation (tg_shape.h), 0 = generic
    TgStagePlan ls, der, qp;
    int staged;             // QP stage: persistent state staged through shared memory
    int slices;             // independent slices of a chunk of at least 8,192 problems (tg_solve_phased)
    size_t np;              // doubles of persistent state per problem
    int chunk;              // problems per chunk (the batch is solved in chunks)
    size_t phased_bytes;
    // scratch of the QP / line-search and derivative stages in workspace slots instead of shared memory; the stages
    // run one after the other on one stream, so they share the slots: `slots` of the stage with more lane groups,
    // `slot_bytes` of the larger need (multiple of 256)
    int slots;
    size_t slot_bytes;
};

#define TG_PHASED_CHUNK_BYTES ((size_t)6 << 30)     // cap of the global state per chunk (the batch is solved in chunks)

static int tg_plan_solve(const TgShape &S, int B, TgSolvePlan *P)
{
    int rc = tg_device_check();
    if (rc) return rc;
    const TgLayout &L = S.L;
    const size_t budget = (size_t)g_smem_optin - 1024;
    const size_t sm_total = 227 * 1024;
    P->fix = tg_plan_fix(S);
    P->np = tg_sqp_persistent_doubles(L);
    // line search: smallest group that leaves >= 8 resident warps' worth of shared memory per SM
    // (shapes with more than 32 variables: 16 lanes at least -- C4 fits 8-lane groups since its derivative stage stages
    // less, but runs 3 % slower with them)
    int gs = tg_env_gs("TG_LS_GS", L.n > 32 && tg_default_gs(L) < 16 ? 16 : tg_default_gs(L));
    while (tg_ls_smem_bytes(L, gs) * 2 > sm_total - 2048 && gs < 32) gs *= 2;
    // shapes whose share does not fit (TG_LS_FAR=1: any shape, for A/B runs): parameters and state prefix read in place,
    // evaluation scratch in workspace slots, 32 lanes per problem
    const char *lsf = getenv("TG_LS_FAR");
    const int ls_far = tg_ls_smem_bytes(L, gs) > budget || (lsf && atoi(lsf) != 0);
    if (ls_far) gs = 32;
    // (the derivative stage stages less than the line search: shared memory of its own)
    P->ls = {gs, ls_far, ls_far ? 0 : tg_ls_smem_bytes(L, gs)};
    P->der = {gs, ls_far, ls_far ? 0 : tg_fd_smem_bytes(L, gs)};
    // QP: lanes per problem from the variables of the subproblem after the elimination of the terminal location rows
    // (tg_sqp_qp_dim): 16, one warp, or two warps (64 lanes) beyond 32, so that every lane-strided loop takes one pass.  Persistent state staged through shared memory when 16 problems still fit.
    {
        const char *v = getenv("TG_QP_GS");
        // (16 lanes run with the state in global memory: only shapes with few dense inequality rows, whose copy sits next
        // to the scratch -- C5: 239 ms against 276 ms with 32 lanes; C2, 11 such rows: 184 ms against 176 ms)
        const int nd = L.m - 2 * L.n_sfc - L.meq;
        gs = v ? atoi(v) : (tg_sqp_qp_dim(L) > 32 ? 64 : (tg_sqp_qp_dim(L) > 16 || nd > 4) ? 32 : 16);
        if (!(gs == 16 || gs == 32 || gs == 64)) gs = 32;        // TG_QP_GS: 16, 32 or 64 (the QP kernels there are); else 32
    }
    const size_t with_state = tg_qp_smem_bytes(L, gs, 1), without = tg_qp_smem_bytes(L, gs, 0);
    // (16-lane groups: 8 problems per CTA, never staged by this rule -- measured: C5 239 ms unstaged, 260 ms staged)
    P->staged = with_state * 4 <= sm_total - 4096;
    if (const char *v = getenv("TG_QP_STAGED")) P->staged = atoi(v) != 0 && with_state <= budget;      // tuning override
    // shapes whose scratch does not fit even unstaged (TG_QP_FAR=1: any shape, for A/B runs): scratch in workspace
    // slots, state in global memory, 64 lanes per problem
    const char *qpf = getenv("TG_QP_FAR");
    const int qp_far = (P->staged ? with_state : without) > budget || (qpf && atoi(qpf) != 0);
    if (qp_far) { gs = 64; P->staged = 0; }
    P->qp = {gs, qp_far, qp_far ? 0 : P->staged ? with_state : without};
    // (a state of tens of MB per problem -- 3-D, N = 512 -- makes chunks of fewer than 1024 problems: the cap holds)
    size_t chunk = TG_PHASED_CHUNK_BYTES / (P->np * sizeof(double));
    if (chunk < 1) chunk = 1;
    if (chunk > (size_t)B) chunk = (size_t)B;
    P->chunk = (int)chunk;
    P->phased_bytes = chunk * P->np * sizeof(double);
    // workspace slots: one per lane group of a grid capped at TG_FAR_CTAS_PER_SM CTAs per SM and at the chunk's work
    auto slots_of = [&](int groups) {
        const size_t need = (chunk + groups - 1) / groups, cap = (size_t)g_sm_count * TG_FAR_CTAS_PER_SM;
        return (need < cap ? need : cap) * groups;
    };
    const size_t qp_slots = qp_far ? slots_of(TG_CTA_THREADS / 64) : 0, ls_slots = ls_far ? slots_of(TG_CTA_THREADS / 32) : 0;
    const size_t qp_bytes = qp_slots * tg_sqp_qp_scratch_doubles(L) * sizeof(double);
    const size_t ls_bytes = ls_slots * tg_sqp_ls_slot_doubles(L) * sizeof(double);
    P->slots = (int)(qp_slots > ls_slots ? qp_slots : ls_slots);
    P->slot_bytes = ((qp_bytes > ls_bytes ? qp_bytes : ls_bytes) + 255) & ~(size_t)255;
    // slices: measured on B200 (65,536 problems): two slices -9.5 % on C2 (short stage kernels, a long tail of rounds
    // with few problems), -2 % on C3, +3 % on C5a, +8 % on C4 (state in L2 / HBM): two when the state is staged in shared
    // memory.  Far-placed shapes run as one slice: the workspace slots serve one grid at a time.
    P->slices = P->staged ? 2 : 1;
    if (const char *v = getenv("TG_SLICES")) P->slices = atoi(v);
    if (P->slot_bytes) P->slices = 1;
    if (P->slices < 1) P->slices = 1;
    if (P->slices > TG_MAX_SLICES) P->slices = TG_MAX_SLICES;
    return 0;
}

// device bookkeeping in front of the per-problem state: [TgRoundCtl x TG_MAX_SLICES | list0[chunk] | list1[chunk] |
// workspace slots (far-placed stages only)]
#define TG_HEADER_BYTES (TG_MAX_SLICES * TG_ROUNDCTL_BYTES)
static size_t tg_lists_bytes(int chunk) { return (((size_t)2 * chunk * sizeof(int)) + 255) & ~(size_t)255; }

// bytes of the solve workspace: the lock-step solve's, or the fused kernel's global workspace where that is larger
static size_t tg_workspace_bytes(const TgShape &S, int B, const TgSolvePlan &P)
{
    const size_t phased = P.phased_bytes + tg_lists_bytes(P.chunk) + P.slot_bytes;
    const size_t fused = tg_fused_workspace_bytes(S, B, g_sm_count, g_smem_optin);
    return (fused > phased ? fused : phased) + TG_HEADER_BYTES;
}

extern "C" size_t tg_solve_workspace_bytes(const int *spec, int B)
{
    TgShape S;
    TgSolvePlan P;
    if (tg_make_shape(spec, &S) || tg_plan_solve(S, B, &P)) return 0;
    return tg_workspace_bytes(S, B, P);
}

extern "C" int tg_solve_plan_info(const int *spec, int B, int *out, int cap)
{
    TgShape S;
    TgSolvePlan P;
    int rc = tg_make_shape(spec, &S);
    if (!rc) rc = tg_plan_solve(S, B > 0 ? B : 1, &P);
    if (rc) return -rc;
    const int v[7] = {P.ls.lanes, P.qp.lanes, P.staged, P.qp.far, P.ls.far, P.slots, (int)(P.slot_bytes >> 10)};
    for (int i = 0; i < 7 && out && i < cap; i++) out[i] = v[i];
    return 7;
}

#define TG_LAUNCH(call, what)                                                   \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        g_launches++;                                                           \
        if (e_ != cudaSuccess) return tg_fail(100 + (int)e_, what, e_);         \
    } while (0)

// ---------------------------------------------------------------------------
// optional per-stage device timing of the lock-step solve (bench.py's roofline): CUDA events on the launching
// stream around every stage launch.  Off by default; the numbers describe the last solve of the calling thread.
// ---------------------------------------------------------------------------
#include <vector>
struct TgSolveStats {
    double ms_ls, ms_qp, flops_qp;
    int launches_ls, launches_qp, rounds;
};
static thread_local TgSolveStats g_stats = {0, 0, 0, 0, 0, 0};
static std::atomic<int> g_stage_timing{0};

extern "C" void tg_set_stage_timing(int on) { g_stage_timing = on; }

extern "C" int tg_last_solve_stats(double *out, int cap)
{
    const double v[6] = {g_stats.ms_ls, g_stats.ms_qp, g_stats.flops_qp, (double)g_stats.launches_ls,
                         (double)g_stats.launches_qp, (double)g_stats.rounds};
    for (int i = 0; i < 6 && i < cap; i++) out[i] = v[i];
    return 6;
}

// A chunk is solved as up to TG_MAX_SLICES independent slices (the plan's count), each with its own round bookkeeping
// and its own stream: while one slice's stage kernel drains (a round lasts as long as its slowest problem), the other
// slices' kernels fill the machine.  Stage timing runs one slice (unoverlapped kernels).
struct TgSliceStreams {
    cudaStream_t st[TG_MAX_SLICES] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t fork = nullptr, join[TG_MAX_SLICES] = {nullptr, nullptr, nullptr, nullptr};
    bool ready = false;
    cudaError_t init()
    {
        if (ready) return cudaSuccess;
        cudaError_t e;
        if ((e = cudaEventCreateWithFlags(&fork, cudaEventDisableTiming))) return e;
        for (int i = 0; i < TG_MAX_SLICES; i++) {
            if ((e = cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking))) return e;
            if ((e = cudaEventCreateWithFlags(&join[i], cudaEventDisableTiming))) return e;
        }
        ready = true;
        return cudaSuccess;
    }
};
// pool of stream sets per device: a solve borrows one for its duration (worker threads of tg_solve_mixed_host come
// and go, so nothing is tied to a thread and nothing leaks)
static std::mutex g_slice_mutex;
static std::vector<TgSliceStreams *> g_slice_free[TG_MAX_DEVICES];
struct TgSliceLease {
    TgSliceStreams *s = nullptr;
    int dev = 0;
    cudaError_t acquire()
    {
        if (s) return cudaSuccess;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        {
            std::lock_guard<std::mutex> lock(g_slice_mutex);
            if (!g_slice_free[dev].empty()) { s = g_slice_free[dev].back(); g_slice_free[dev].pop_back(); }
        }
        if (!s) s = new TgSliceStreams();
        return s->init();
    }
    ~TgSliceLease()
    {
        if (!s) return;
        std::lock_guard<std::mutex> lock(g_slice_mutex);
        g_slice_free[dev].push_back(s);
    }
};

// the plan's stage: its launcher for its lanes, its shared memory and slots
static cudaError_t tg_launch_stage(const TgStageLauncher launchers[4], const TgStagePlan &s, TgStageLaunch &a, double *slots)
{
    a.smem = s.smem;
    a.far = s.far ? slots : nullptr;
    const TgStageLauncher launch = launchers[tg_lanes_index(s.lanes)];
    assert(launch);
    return launch(a);
}

static int tg_solve_phased(const TgShape &S, const TgSolvePlan &P, int B, const double *par, double *x, double *f,
                           int *status, int *nit, int *violation, double *lam, double *kkt, int maxiter, double ftol,
                           int flags, void *workspace, cudaStream_t st)
{
    const TgLayout &L = S.L;
    char *wsb = (char *)workspace;
    int *list_base = (int *)(wsb + TG_HEADER_BYTES);
    double *slots = (double *)(wsb + TG_HEADER_BYTES + tg_lists_bytes(P.chunk));
    double *pws_base = (double *)((char *)slots + P.slot_bytes);
    const bool timing = g_stage_timing.load() != 0;
    std::vector<cudaEvent_t> ev;
    if (timing) g_stats = TgSolveStats{0, 0, 0, 0, 0, 0};
    auto mark = [&]() -> cudaError_t {
        if (!timing) return cudaSuccess;
        cudaEvent_t e;
        cudaError_t rc_ = cudaEventCreate(&e);
        if (rc_ != cudaSuccess) return rc_;
        ev.push_back(e);
        return cudaEventRecord(e, st);
    };
    TgSliceLease lease;
    for (int lo = 0; lo < B; lo += P.chunk) {
        const int nbc = B - lo < P.chunk ? B - lo : P.chunk;
        const int ns = (timing || nbc < 8192) ? 1 : P.slices;
        if (ns > 1) {
            TG_CUDA(lease.acquire());
            TG_CUDA(cudaEventRecord(lease.s->fork, st));
        }
        TgSliceStreams *const ss = lease.s;          // only touched when ns > 1
        struct Slice { int lo, nb, done; TgRoundCtl *rc; int *lists[2]; double *pws; cudaStream_t st; } sl[TG_MAX_SLICES];
        for (int k = 0; k < ns; k++) {
            Slice &q = sl[k];
            q.lo = (int)((long long)nbc * k / ns);
            q.nb = (int)((long long)nbc * (k + 1) / ns) - q.lo;
            q.done = 0;
            q.rc = (TgRoundCtl *)(wsb + (size_t)k * TG_ROUNDCTL_BYTES);
            q.lists[0] = list_base + q.lo;
            q.lists[1] = list_base + P.chunk + q.lo;
            q.pws = pws_base + (size_t)q.lo * P.np;
            q.st = ns > 1 ? ss->st[k] : st;
            if (ns > 1) TG_CUDA(cudaStreamWaitEvent(q.st, ss->fork, 0));
            TG_CUDA(cudaMemsetAsync(q.rc, 0, TG_ROUNDCTL_BYTES, q.st));
            TG_LAUNCH(tg_launch_begin_g32(S, q.nb, x + (size_t)(lo + q.lo) * L.n, q.pws, P.np, maxiter, ftol, flags, q.rc,
                                          q.lists[0], q.st), "tg_sqp_begin_kernel");
        }
        // each round = one SLSQP major iteration of every unfinished problem; maxiter + 1 rounds finish everything.
        // Round r works through list r & 1; the QP stage builds the other list from the problems still running.
        for (int round = 0; round <= maxiter + 1; round++) {
            const int par_ = round & 1;
            bool any = false;
            for (int k = 0; k < ns; k++) {
                Slice &q = sl[k];
                if (q.done >= q.nb) continue;
                any = true;
                TgStageLaunch a = {S, q.nb, par + (size_t)(lo + q.lo) * L.P, q.pws, P.np, 0, nullptr, P.staged, q.rc,
                                   q.lists[par_], q.lists[par_ ^ 1], par_, g_sm_count, P.fix, q.st};
                TG_CUDA(mark());
                TG_LAUNCH(tg_launch_stage(tg_ls_launchers, P.ls, a, slots), "tg_sqp_ls_kernel");
                TG_LAUNCH(tg_launch_stage(tg_fd_launchers, P.der, a, slots), "tg_sqp_der_kernel");
                TG_CUDA(mark());
                TG_LAUNCH(tg_launch_stage(tg_qp_launchers, P.qp, a, slots), "tg_sqp_qp_kernel");
                TG_CUDA(mark());
            }
            if (!any) break;
            if (timing) g_stats.rounds++;
            if ((round & 7) == 7) {      // poll the number of finished problems
                for (int k = 0; k < ns; k++)
                    if (sl[k].done < sl[k].nb)
                        TG_CUDA(cudaMemcpyAsync(&sl[k].done, &sl[k].rc->done, sizeof(int), cudaMemcpyDeviceToHost, sl[k].st));
                for (int k = 0; k < ns; k++) TG_CUDA(cudaStreamSynchronize(sl[k].st));
            }
        }
        for (int k = 0; k < ns; k++) {
            Slice &q = sl[k];
            const int o = lo + q.lo;
            TG_LAUNCH(tg_launch_finish_g32(S, q.nb, q.pws, P.np, x + (size_t)o * L.n, f ? f + o : nullptr, status ? status + o : nullptr,
                                           nit ? nit + o : nullptr, violation ? violation + o : nullptr,
                                           lam ? lam + (size_t)o * L.m : nullptr, kkt ? kkt + (size_t)o * 4 : nullptr, q.rc, q.st),
                      "tg_sqp_finish_kernel");
            if (ns > 1) {
                TG_CUDA(cudaEventRecord(ss->join[k], q.st));
                TG_CUDA(cudaStreamWaitEvent(st, ss->join[k], 0));
            }
        }
        if (timing) {
            double fl = 0;
            TG_CUDA(cudaMemcpyAsync(&fl, &sl[0].rc->flops_qp, sizeof(double), cudaMemcpyDeviceToHost, st));
            TG_CUDA(cudaStreamSynchronize(st));
            g_stats.flops_qp += fl;
            const bool dump = getenv("TG_DUMP_ROUNDS") != nullptr;
            for (size_t k = 0; k + 3 <= ev.size(); k += 3) {
                float a = 0, b = 0;
                cudaEventElapsedTime(&a, ev[k], ev[k + 1]);
                cudaEventElapsedTime(&b, ev[k + 1], ev[k + 2]);
                if (dump) fprintf(stderr, "round %3zu: ls+fd %.3f ms  qp %.3f ms\n", k / 3, a, b);
                g_stats.ms_ls += a; g_stats.ms_qp += b;
                g_stats.launches_ls++; g_stats.launches_qp++;
            }
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
            ev.clear();
        }
    }
    return 0;
}

extern "C" int tg_solve_batch_kkt(const int *spec, int B, const double *par, double *x, double *f, int *status, int *nit,
                                  int *violation, int maxiter, double ftol, int flags, void *workspace,
                                  size_t workspace_bytes, void *stream, double *lam, double *kkt)
{
    TgShape S;
    TgSolvePlan P;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if ((rc = tg_plan_solve(S, B, &P))) return rc;
    if (!workspace || workspace_bytes < tg_workspace_bytes(S, B, P)) return tg_fail(4, "workspace too small (see tg_solve_workspace_bytes)");
    cudaStream_t st = (cudaStream_t)stream;
    if (flags & TG_SOLVE_FUSED) {
        int *counters = (int *)workspace;
        TG_CUDA(cudaMemsetAsync(counters, 0, 256, st));
        TG_LAUNCH(tg_launch_fused_g32(S, B, par, x, f, status, nit, violation, lam, kkt, maxiter, ftol, flags, (char *)workspace + 256,
                                      counters, g_sm_count, g_smem_optin, st), "tg_solve_kernel");
        return 0;
    }
    return tg_solve_phased(S, P, B, par, x, f, status, nit, violation, lam, kkt, maxiter, ftol, flags, workspace, st);
}

extern "C" int tg_solve_batch(const int *spec, int B, const double *par, double *x, double *f, int *status, int *nit,
                              int *violation, int maxiter, double ftol, int flags, void *workspace,
                              size_t workspace_bytes, void *stream)
{
    return tg_solve_batch_kkt(spec, B, par, x, f, status, nit, violation, maxiter, ftol, flags, workspace, workspace_bytes,
                              stream, nullptr, nullptr);
}

// ---------------------------------------------------------------------------
// measured FP64 peak of this device (denominator of the solve kernels' roofline): 8 independent DFMA chains per
// thread, every SM full.  Returns TFLOP/s (2 flops per DFMA).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tg_fp64_peak_kernel(double *out, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-9;
    #pragma unroll 1
    for (int i = 0; i < iters; i++) {
        #pragma unroll
        for (int r = 0; r < 8; r++) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" int tg_measure_fp64_peak(double *tflops)
{
    int rc = tg_device_check();
    if (rc) return rc;
    if (!tflops) return tg_fail(1, "tflops is NULL");
    const int ctas = g_sm_count * 8, threads = 256, iters = 4096;
    double *buf = nullptr;
    TG_CUDA(cudaMalloc(&buf, (size_t)ctas * threads * sizeof(double)));
    cudaEvent_t a, b;
    TG_CUDA(cudaEventCreate(&a));
    TG_CUDA(cudaEventCreate(&b));
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
        TG_CUDA(cudaEventRecord(a, 0));
        tg_fp64_peak_kernel<<<ctas, threads>>>(buf, iters, 1.0 + rep);
        TG_CUDA(cudaEventRecord(b, 0));
        TG_CUDA(cudaEventSynchronize(b));
        float ms = 0;
        TG_CUDA(cudaEventElapsedTime(&ms, a, b));
        const double tf = 2.0 * 64.0 * iters * (double)ctas * threads / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    g_launches += 4;
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(buf);
    *tflops = best;
    return 0;
}

// ---------------------------------------------------------------------------
// host-buffer entry points
// ---------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return tg_fail(100 + (int)e, "cudaMalloc", e);
        cap = bytes;
        return 0;
    }
};
// cached device buffers of the host-buffer entry points, one set per device (callers on different devices do not
// serialise against each other; callers on the same device do)
struct TgHostCtx {
    std::mutex mu;
    DevBuf par, x, f, g, c, j, i, ws;
    cudaStream_t st[2] = {nullptr, nullptr};      // chunk pipeline of tg_eval_host
};
static TgHostCtx g_host[TG_MAX_DEVICES];
static TgHostCtx *tg_host_ctx()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= TG_MAX_DEVICES) return nullptr;
    return &g_host[dev];
}

// true when every non-NULL pointer is page-locked host memory (cudaHostAlloc / cudaHostRegister / torch pin_memory):
// such buffers are copied by the DMA engines asynchronously, so chunks of a batch can overlap their copies and kernels
static bool tg_all_pinned(std::initializer_list<const void *> ptrs)
{
    for (const void *p : ptrs) {
        if (!p) continue;
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
        if (a.type != cudaMemoryTypeHost) return false;
    }
    return true;
}

#define TG_HOST_CHUNKS 8          // pipeline depth of the host-buffer entry points on page-locked buffers

extern "C" int tg_eval_host(const int *spec, int B, const double *par, const double *x, double *f, double *g, double *c,
                            double *jnl)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if ((rc = tg_device_check())) return rc;
    TgHostCtx *H = tg_host_ctx();
    if (!H) return tg_fail(10, "cannot identify the current device");
    std::lock_guard<std::mutex> lock(H->mu);
    DevBuf &g_par = H->par, &g_x = H->x, &g_f = H->f, &g_g = H->g, &g_c = H->c, &g_j = H->j;
    const TgLayout &L = S.L;
    const size_t nb = sizeof(double);
    if ((rc = g_par.ensure((size_t)B * (L.P + 1) * nb)) || (rc = g_x.ensure((size_t)B * L.n * nb))) return rc;
    if (f && (rc = g_f.ensure((size_t)B * nb))) return rc;
    if (g && (rc = g_g.ensure((size_t)B * L.n * nb))) return rc;
    if (c && (rc = g_c.ensure((size_t)B * (L.m + 1) * nb))) return rc;
    if (jnl && (rc = g_j.ensure((size_t)B * (L.m_nl * L.n + 1) * nb))) return rc;
    // Page-locked caller buffers: the batch goes through in chunks on two streams, so the upload of one chunk, the
    // kernel of another and the download of a third (the dense Jacobian rows: ~85 % of the bytes) overlap.  Pageable
    // buffers are staged by the driver synchronously: one chunk.
    const bool pinned = B >= 4096 && tg_all_pinned({par, x, f, g, c, jnl});
    const int chunks = pinned ? TG_HOST_CHUNKS : 1;
    cudaStream_t st[2] = {0, 0};
    if (pinned) {
        for (int k = 0; k < 2; k++) {
            if (!H->st[k]) TG_CUDA(cudaStreamCreateWithFlags(&H->st[k], cudaStreamNonBlocking));
            st[k] = H->st[k];
        }
    }
    for (int k = 0; k < chunks; k++) {
        const size_t lo = (size_t)B * k / chunks, hi = (size_t)B * (k + 1) / chunks, cnt = hi - lo;
        if (!cnt) continue;
        cudaStream_t s = st[k & 1];
        double *dpar = (double *)g_par.p + lo * L.P, *dx = (double *)g_x.p + lo * L.n;
        double *df = f ? (double *)g_f.p + lo : nullptr, *dg = g ? (double *)g_g.p + lo * L.n : nullptr;
        double *dc = c ? (double *)g_c.p + lo * L.m : nullptr, *dj = jnl ? (double *)g_j.p + lo * L.m_nl * L.n : nullptr;
        TG_CUDA(cudaMemcpyAsync(dpar, par + lo * L.P, cnt * L.P * nb, cudaMemcpyHostToDevice, s));
        TG_CUDA(cudaMemcpyAsync(dx, x + lo * L.n, cnt * L.n * nb, cudaMemcpyHostToDevice, s));
        if ((rc = tg_eval_batch(spec, (int)cnt, dpar, dx, df, dg, dc, dj, s))) return rc;
        if (f) TG_CUDA(cudaMemcpyAsync(f + lo, df, cnt * nb, cudaMemcpyDeviceToHost, s));
        if (g) TG_CUDA(cudaMemcpyAsync(g + lo * L.n, dg, cnt * L.n * nb, cudaMemcpyDeviceToHost, s));
        if (c) TG_CUDA(cudaMemcpyAsync(c + lo * L.m, dc, cnt * L.m * nb, cudaMemcpyDeviceToHost, s));
        if (jnl) TG_CUDA(cudaMemcpyAsync(jnl + lo * L.m_nl * L.n, dj, cnt * L.m_nl * L.n * nb, cudaMemcpyDeviceToHost, s));
    }
    TG_CUDA(cudaStreamSynchronize(st[0]));
    if (pinned) TG_CUDA(cudaStreamSynchronize(st[1]));
    return 0;
}

extern "C" int tg_solve_host(const int *spec, int B, const double *par, double *x, double *f, int *status, int *nit,
                             int *violation, int maxiter, double ftol, int flags)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if ((rc = tg_device_check())) return rc;
    TgHostCtx *H = tg_host_ctx();
    if (!H) return tg_fail(10, "cannot identify the current device");
    std::lock_guard<std::mutex> lock(H->mu);
    DevBuf &g_par = H->par, &g_x = H->x, &g_f = H->f, &g_i = H->i, &g_ws = H->ws;
    const TgLayout &L = S.L;
    const size_t nb = sizeof(double);
    const size_t wsb = tg_solve_workspace_bytes(spec, B);
    if (wsb == 0) return tg_fail(5, g_err[0] ? g_err : "cannot plan the solve kernel");
    if ((rc = g_par.ensure((size_t)B * (L.P + 1) * nb)) || (rc = g_x.ensure((size_t)B * L.n * nb)) ||
        (rc = g_f.ensure((size_t)B * nb)) || (rc = g_i.ensure((size_t)B * 3 * sizeof(int))) || (rc = g_ws.ensure(wsb)))
        return rc;
    int *di = (int *)g_i.p;
    TG_CUDA(cudaMemcpyAsync(g_par.p, par, (size_t)B * L.P * nb, cudaMemcpyHostToDevice, 0));
    TG_CUDA(cudaMemcpyAsync(g_x.p, x, (size_t)B * L.n * nb, cudaMemcpyHostToDevice, 0));
    rc = tg_solve_batch(spec, B, (const double *)g_par.p, (double *)g_x.p, (double *)g_f.p, di, di + B, di + 2 * B,
                        maxiter, ftol, flags, g_ws.p, wsb, 0);
    if (rc) return rc;
    TG_CUDA(cudaMemcpyAsync(x, g_x.p, (size_t)B * L.n * nb, cudaMemcpyDeviceToHost, 0));
    if (f) TG_CUDA(cudaMemcpyAsync(f, g_f.p, (size_t)B * nb, cudaMemcpyDeviceToHost, 0));
    if (status) TG_CUDA(cudaMemcpyAsync(status, di, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, 0));
    if (nit) TG_CUDA(cudaMemcpyAsync(nit, di + B, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, 0));
    if (violation) TG_CUDA(cudaMemcpyAsync(violation, di + 2 * B, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, 0));
    TG_CUDA(cudaStreamSynchronize(0));
    return 0;
}

// ---------------------------------------------------------------------------
// f3 (SURVEY.md 8(f)): problems of DIFFERENT shapes in one call.  The reference chooses the number of control
// points and the corridor split from the geometry (TG/trajectory_generator.py:148-162), so a real workload is a
// mix of shapes.  The caller hands over the buckets (problems grouped by shape descriptor); up to
// TG_MIXED_WORKERS buckets are in flight at a time, each on its own stream with its own device buffers, so that
// the lock-step rounds of one bucket fill the SMs that the tail of another bucket's round leaves idle.
// ---------------------------------------------------------------------------
#define TG_MIXED_WORKERS 4

struct TgMixedSlot {
    cudaStream_t st = nullptr;
    DevBuf par, x, f, i, ws;
};
struct TgMixedCtx {
    std::mutex mu;
    TgMixedSlot slot[TG_MIXED_WORKERS];
};
static TgMixedCtx g_mixed_ctx[TG_MAX_DEVICES];

// shared by tg_solve_mixed_host (host buffers: copies on the bucket's stream) and tg_solve_mixed_batch (device
// pointers: the buckets' streams fork from and join the caller's stream)
static int tg_solve_mixed_impl(bool host, int nbuckets, const int *specs, const int *counts, const double *const *par,
                               double *const *x, double *const *f, int *const *status, int *const *nit,
                               int *const *violation, double *const *lam, double *const *kkt, int maxiter, double ftol,
                               int flags, cudaStream_t caller)
{
    if (nbuckets <= 0) return 0;
    if (!specs || !counts || !par || !x) return tg_fail(1, "tg_solve_mixed: NULL argument");
    int rc = tg_device_check();
    if (rc) return rc;
    int dev = 0;
    TG_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= TG_MAX_DEVICES) return tg_fail(10, "device index out of range");
    std::lock_guard<std::mutex> lock(g_mixed_ctx[dev].mu);
    TgMixedSlot *const g_mixed = g_mixed_ctx[dev].slot;
    // validate every bucket before any work is queued
    for (int k = 0; k < nbuckets; k++) {
        TgShape S;
        if ((rc = tg_make_shape(specs + (size_t)k * TG_SP_COUNT, &S))) return rc;
        if (counts[k] > 0 && (!par[k] || !x[k])) return tg_fail(1, "tg_solve_mixed: NULL bucket buffer");
    }
    const int workers = nbuckets < TG_MIXED_WORKERS ? nbuckets : TG_MIXED_WORKERS;
    for (int w = 0; w < workers; w++)
        if (!g_mixed[w].st) TG_CUDA(cudaStreamCreateWithFlags(&g_mixed[w].st, cudaStreamNonBlocking));
    // every slot is sized for the largest bucket up front: which worker takes which bucket varies from call to call, and
    // a slot that had to grow in the middle of a call (cudaFree + cudaMalloc synchronise the device) cost up to 2.5x
    {
        size_t ws_max = 0, par_max = 0, x_max = 0, f_max = 0, i_max = 0;
        for (int k = 0; k < nbuckets; k++) {
            if (counts[k] <= 0) continue;
            const int *spec = specs + (size_t)k * TG_SP_COUNT;
            TgShape S;
            tg_make_shape(spec, &S);
            const size_t B = (size_t)counts[k], wsb = tg_solve_workspace_bytes(spec, counts[k]);
            if (!wsb) return tg_fail(5, g_err[0] ? g_err : "cannot plan the solve kernel");
            ws_max = wsb > ws_max ? wsb : ws_max;
            par_max = B * (S.L.P + 1) * sizeof(double) > par_max ? B * (S.L.P + 1) * sizeof(double) : par_max;
            x_max = B * S.L.n * sizeof(double) > x_max ? B * S.L.n * sizeof(double) : x_max;
            f_max = B * sizeof(double) > f_max ? B * sizeof(double) : f_max;
            i_max = B * 3 * sizeof(int) > i_max ? B * 3 * sizeof(int) : i_max;
        }
        for (int w = 0; w < workers; w++) {
            if ((rc = g_mixed[w].ws.ensure(ws_max))) return rc;
            if (host && ((rc = g_mixed[w].par.ensure(par_max)) || (rc = g_mixed[w].x.ensure(x_max)) ||
                         (rc = g_mixed[w].f.ensure(f_max)) || (rc = g_mixed[w].i.ensure(i_max)))) return rc;
        }
    }
    cudaEvent_t fork = nullptr;
    if (!host) {
        TG_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
        TG_CUDA(cudaEventRecord(fork, caller));
        for (int w = 0; w < workers; w++) TG_CUDA(cudaStreamWaitEvent(g_mixed[w].st, fork, 0));
    }
    // largest buckets first: the long solves start early and the small ones fill in around them
    std::vector<int> order(nbuckets);
    for (int k = 0; k < nbuckets; k++) order[k] = k;
    for (int a = 1; a < nbuckets; a++)
        for (int b = a; b > 0 && counts[order[b]] > counts[order[b - 1]]; b--) { int t = order[b]; order[b] = order[b - 1]; order[b - 1] = t; }
    std::atomic<int> cursor{0};
    std::vector<int> rcs(workers, 0);
    std::vector<std::string> errs(workers);
    auto work = [&](int w) {
        cudaSetDevice(dev);
        TgMixedSlot &s = g_mixed[w];
        for (;;) {
            const int at = cursor.fetch_add(1);
            if (at >= nbuckets) break;
            const int k = order[at], B = counts[k];
            if (B <= 0) continue;
            const int *spec = specs + (size_t)k * TG_SP_COUNT;
            TgShape S;
            tg_make_shape(spec, &S);
            const TgLayout &L = S.L;
            const size_t nb = sizeof(double);
            const size_t wsb = tg_solve_workspace_bytes(spec, B);
            int r = wsb ? 0 : tg_fail(5, g_err[0] ? g_err : "cannot plan the solve kernel");
            if (!r) r = s.ws.ensure(wsb);
            if (host) {
                if (!r) r = s.par.ensure((size_t)B * (L.P + 1) * nb);
                if (!r) r = s.x.ensure((size_t)B * L.n * nb);
                if (!r) r = s.f.ensure((size_t)B * nb);
                if (!r) r = s.i.ensure((size_t)B * 3 * sizeof(int));
            }
            int *di = (int *)s.i.p;
            auto cp = [&](void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
                if (r) return;
                cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, s.st);
                if (e != cudaSuccess) r = tg_fail(100 + (int)e, "cudaMemcpyAsync", e);
            };
            if (host) {
                cp(s.par.p, par[k], (size_t)B * L.P * nb, cudaMemcpyHostToDevice);
                cp(s.x.p, x[k], (size_t)B * L.n * nb, cudaMemcpyHostToDevice);
                if (!r) r = tg_solve_batch(spec, B, (const double *)s.par.p, (double *)s.x.p, (double *)s.f.p, di, di + B, di + 2 * B,
                                           maxiter, ftol, flags, s.ws.p, wsb, s.st);
                cp(x[k], s.x.p, (size_t)B * L.n * nb, cudaMemcpyDeviceToHost);
                if (f && f[k]) cp(f[k], s.f.p, (size_t)B * nb, cudaMemcpyDeviceToHost);
                if (status && status[k]) cp(status[k], di, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost);
                if (nit && nit[k]) cp(nit[k], di + B, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost);
                if (violation && violation[k]) cp(violation[k], di + 2 * B, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost);
            } else if (!r) {
                r = tg_solve_batch_kkt(spec, B, par[k], x[k], f ? f[k] : nullptr, status ? status[k] : nullptr,
                                       nit ? nit[k] : nullptr, violation ? violation[k] : nullptr, maxiter, ftol, flags, s.ws.p,
                                       wsb, s.st, lam ? lam[k] : nullptr, kkt ? kkt[k] : nullptr);
            }
            // (the slot's workspace and staging buffers are reused by this worker's next bucket, which is queued on the
            // same stream; host buffers must be complete before the call returns)
            cudaError_t e = host ? cudaStreamSynchronize(s.st) : cudaSuccess;
            if (!r && e != cudaSuccess) r = tg_fail(100 + (int)e, "cudaStreamSynchronize", e);
            if (r) { rcs[w] = r; errs[w] = g_err; break; }
        }
    };
    std::vector<std::thread> pool;
    for (int w = 1; w < workers; w++) pool.emplace_back(work, w);
    work(0);
    for (std::thread &t : pool) t.join();
    if (!host) {
        // the caller's stream continues after every bucket's stream
        for (int w = 0; w < workers; w++) {
            cudaEventRecord(fork, g_mixed[w].st);
            cudaStreamWaitEvent(caller, fork, 0);
        }
        cudaEventDestroy(fork);
    }
    for (int w = 0; w < workers; w++)
        if (rcs[w]) return tg_fail(rcs[w], errs[w].c_str());
    return 0;
}

extern "C" int tg_solve_mixed_host(int nbuckets, const int *specs, const int *counts, const double *const *par,
                                   double *const *x, double *const *f, int *const *status, int *const *nit,
                                   int *const *violation, int maxiter, double ftol, int flags)
{
    return tg_solve_mixed_impl(true, nbuckets, specs, counts, par, x, f, status, nit, violation, nullptr, nullptr, maxiter, ftol,
                               flags, nullptr);
}

extern "C" int tg_solve_mixed_batch_kkt(int nbuckets, const int *specs, const int *counts, const double *const *par,
                                        double *const *x, double *const *f, int *const *status, int *const *nit,
                                        int *const *violation, int maxiter, double ftol, int flags, void *stream,
                                        double *const *lam, double *const *kkt)
{
    return tg_solve_mixed_impl(false, nbuckets, specs, counts, par, x, f, status, nit, violation, lam, kkt, maxiter, ftol, flags,
                               (cudaStream_t)stream);
}

extern "C" int tg_solve_mixed_batch(int nbuckets, const int *specs, const int *counts, const double *const *par,
                                    double *const *x, double *const *f, int *const *status, int *const *nit,
                                    int *const *violation, int maxiter, double ftol, int flags, void *stream)
{
    return tg_solve_mixed_batch_kkt(nbuckets, specs, counts, par, x, f, status, nit, violation, maxiter, ftol, flags, stream,
                                    nullptr, nullptr);
}

// ---------------------------------------------------------------------------
// multi-start solves: expansion of B problems into B * K seeded starts (tg_multistart.cu), and the selection of the best
// start per problem after the caller's ordinary solve of the B * K rows (tg_kernels_eval.inc, planned as tg_eval_batch)
// ---------------------------------------------------------------------------
static int tg_multistart_args(const char *what, int B, int K)
{
    if (K < 1) return tg_fail(2, (std::string(what) + ": the number of starts K must be at least 1").c_str());
    if ((long long)B * K > 0x7fffffffLL) return tg_fail(2, (std::string(what) + ": B * K exceeds the int range").c_str());
    return 0;
}

extern "C" int tg_multistart_expand(const int *spec, int B, int K, const double *par, const double *x0,
                                    unsigned long long seed, double spread, double *par_out, double *x_out, void *stream)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc || (rc = tg_multistart_args("tg_multistart_expand", B, K))) return rc;
    if (!(spread >= 0 && spread <= 1e300)) return tg_fail(2, "tg_multistart_expand: spread must be finite and >= 0");
    if (B <= 0) return 0;
    if (!par || !x0 || !par_out || !x_out) return tg_fail(1, "tg_multistart_expand: NULL argument");
    if ((rc = tg_device_check())) return rc;
    cudaError_t e = tg_launch_multistart_expand(S.L, B, K, par, x0, seed, spread, par_out, x_out, g_sm_count, (cudaStream_t)stream);
    g_launches++;
    if (e != cudaSuccess) return tg_fail(100 + (int)e, "tg_multistart_expand_kernel launch", e);
    return 0;
}

extern "C" int tg_multistart_select(const int *spec, int B, int K, const double *par, const double *xs, const double *f,
                                    const int *status, const int *nit, const int *violation, double tol, double *x_best,
                                    double *f_best, int *status_best, int *nit_best, int *violation_best, int *best_start,
                                    double *max_violation, void *stream)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc || (rc = tg_multistart_args("tg_multistart_select", B, K))) return rc;
    if (B <= 0) return 0;
    if (!par || !xs || !f || !status || !nit || !violation || !x_best || !f_best || !status_best || !nit_best ||
        !violation_best || !best_start)
        return tg_fail(1, "tg_multistart_select: NULL argument (only max_violation may be NULL)");
    if ((rc = tg_device_check())) return rc;
    const int gs = tg_env_gs("TG_EVAL_GS", tg_default_gs(S.L));
    const int groups = tg_eval_groups(S.L, gs, true, g_smem_optin);
    const size_t need = (size_t)tg_eval_group_doubles(S.L, true) * sizeof(double);
    if (groups == 0) {
        snprintf(g_err, sizeof g_err, "tg_select_kernel: a problem with n = %d, m = %d needs %zu bytes of shared memory, "
                 "more than the device's %d", S.L.n, S.L.m, need, g_smem_optin);
        return 3;
    }
    int grid = (B + groups - 1) / groups;
    if (grid > g_sm_count * 32) grid = g_sm_count * 32;
    const TgSelectLaunch a = {S, B, K, par, xs, f, status, nit, violation, tol, x_best, f_best, status_best, nit_best,
                              violation_best, best_start, max_violation, tg_plan_fix(S), grid, groups, groups * need,
                              (cudaStream_t)stream};
    static cudaError_t (*const launchers[3])(const TgSelectLaunch &) = {tg_launch_select_g8, tg_launch_select_g16, tg_launch_select_g32};
    cudaError_t e = launchers[tg_lanes_index(gs)](a);
    g_launches++;
    if (e != cudaSuccess) return tg_fail(100 + (int)e, "tg_select_kernel launch", e);
    return 0;
}

// ---------------------------------------------------------------------------
// post-solve polish (tg_kernels_polish.inc) and parameter sensitivities (tg_kernels_sens.inc): lanes from the shape,
// lane groups per CTA from shared memory; shapes whose per-problem scratch (`per_doubles`: tg_polish_group_doubles or
// tg_sens_group_doubles) does not fit (or TG_POLISH_FAR=1) take it from workspace slots, one per lane group of a grid
// capped at TG_FAR_CTAS_PER_SM CTAs per SM and at TG_POLISH_FAR_BYTES of slots.  Near and far use the same lanes, so
// that they compute the same bits.
// ---------------------------------------------------------------------------
#define TG_POLISH_FAR_BYTES ((size_t)4 << 30)
struct TgPolishPlan {
    int fix, lanes, far, groups, grid;
    size_t per_bytes, smem, ws_bytes;
};

static int tg_plan_polish(const TgShape &S, int B, size_t per_doubles, TgPolishPlan *P)
{
    int rc = tg_device_check();
    if (rc) return rc;
    const TgLayout &L = S.L;
    P->fix = tg_plan_fix(S);
    // (the dense linear algebra strides over the free variables: a warp once they are more than 32)
    P->lanes = L.n > 32 ? 32 : tg_default_gs(L);
    P->per_bytes = per_doubles * sizeof(double);
    const size_t fit = ((size_t)g_smem_optin - 1024) / P->per_bytes;
    const char *v = getenv("TG_POLISH_FAR");
    P->far = fit == 0 || (v && atoi(v) != 0);
    P->groups = TG_CTA_THREADS / P->lanes;
    if (!P->far && fit < (size_t)P->groups) P->groups = (int)fit;
    size_t grid = ((size_t)B + P->groups - 1) / P->groups, cap = (size_t)g_sm_count * 32;
    if (P->far) {
        const size_t cta_bytes = (size_t)P->groups * P->per_bytes, budget = TG_POLISH_FAR_BYTES / cta_bytes;
        cap = (size_t)g_sm_count * TG_FAR_CTAS_PER_SM;
        if (budget < cap) cap = budget > 0 ? budget : 1;
    }
    P->grid = (int)(grid < cap ? grid : cap);
    P->smem = P->far ? 0 : (size_t)P->groups * P->per_bytes;
    P->ws_bytes = P->far ? (((size_t)P->grid * P->groups * P->per_bytes) + 255) & ~(size_t)255 : 0;
    return 0;
}

// the five fields of tg_polish_plan_info / tg_sens_plan_info
static int tg_plan_info_out(const TgPolishPlan &P, int *out, int cap)
{
    const int v[5] = {P.lanes, P.far, P.groups, P.grid, (int)(P.per_bytes >> 10)};
    for (int i = 0; i < 5 && out && i < cap; i++) out[i] = v[i];
    return 5;
}

extern "C" size_t tg_polish_workspace_bytes(const int *spec, int B)
{
    TgShape S;
    TgPolishPlan P;
    if (tg_make_shape(spec, &S) || tg_plan_polish(S, B > 0 ? B : 1, tg_polish_group_doubles(S.L), &P)) return 0;
    return P.ws_bytes;
}

extern "C" int tg_polish_plan_info(const int *spec, int B, int *out, int cap)
{
    TgShape S;
    TgPolishPlan P;
    int rc = tg_make_shape(spec, &S);
    if (!rc) rc = tg_plan_polish(S, B > 0 ? B : 1, tg_polish_group_doubles(S.L), &P);
    if (rc) return -rc;
    return tg_plan_info_out(P, out, cap);
}

extern "C" int tg_polish_batch(const int *spec, int B, const double *par, double *x, double *f, const int *status,
                               int *violation, double *lam, double *kkt, int *polish_status, int *polish_iters,
                               int maxiter, double tol, void *ws, size_t ws_bytes, void *stream)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if (!par || !x || !f || !status || !violation || !lam || !kkt || !polish_status || !polish_iters)
        return tg_fail(1, "tg_polish_batch: NULL argument");
    TgPolishPlan P;
    if ((rc = tg_plan_polish(S, B, tg_polish_group_doubles(S.L), &P))) return rc;
    if (P.ws_bytes && (!ws || ws_bytes < P.ws_bytes)) return tg_fail(4, "workspace too small (see tg_polish_workspace_bytes)");
    const TgPolishLaunch a = {S, B, par, x, f, status, violation, lam, kkt, polish_status, polish_iters, maxiter, tol,
                              P.far ? (double *)ws : nullptr, P.fix, P.grid, P.groups, P.smem, (cudaStream_t)stream};
    static cudaError_t (*const launchers[3])(const TgPolishLaunch &) = {tg_launch_polish_g8, tg_launch_polish_g16, tg_launch_polish_g32};
    cudaError_t e = launchers[tg_lanes_index(P.lanes)](a);
    g_launches++;
    if (e != cudaSuccess) return tg_fail(100 + (int)e, "tg_polish_kernel launch", e);
    return 0;
}

extern "C" size_t tg_sens_workspace_bytes(const int *spec, int B)
{
    TgShape S;
    TgPolishPlan P;
    if (tg_make_shape(spec, &S) || tg_plan_polish(S, B > 0 ? B : 1, tg_sens_group_doubles(S.L), &P)) return 0;
    return P.ws_bytes;
}

extern "C" int tg_sens_plan_info(const int *spec, int B, int *out, int cap)
{
    TgShape S;
    TgPolishPlan P;
    int rc = tg_make_shape(spec, &S);
    if (!rc) rc = tg_plan_polish(S, B > 0 ? B : 1, tg_sens_group_doubles(S.L), &P);
    if (rc) return -rc;
    return tg_plan_info_out(P, out, cap);
}

extern "C" int tg_sens_batch(const int *spec, int B, const double *par, const double *x, const int *status,
                             const double *lam, const double *x_bar, const double *f_bar, double *par_bar,
                             int *sens_status, double tol, void *ws, size_t ws_bytes, void *stream)
{
    TgShape S;
    int rc = tg_make_shape(spec, &S);
    if (rc) return rc;
    if (B <= 0) return 0;
    if (!par || !x || !status || !lam || !x_bar || !par_bar || !sens_status)
        return tg_fail(1, "tg_sens_batch: NULL argument");
    TgPolishPlan P;
    if ((rc = tg_plan_polish(S, B, tg_sens_group_doubles(S.L), &P))) return rc;
    if (P.ws_bytes && (!ws || ws_bytes < P.ws_bytes)) return tg_fail(4, "workspace too small (see tg_sens_workspace_bytes)");
    const TgSensLaunch a = {S, B, par, x, status, lam, x_bar, f_bar, par_bar, sens_status, tol,
                            P.far ? (double *)ws : nullptr, P.fix, P.grid, P.groups, P.smem, (cudaStream_t)stream};
    static cudaError_t (*const launchers[3])(const TgSensLaunch &) = {tg_launch_sens_g8, tg_launch_sens_g16, tg_launch_sens_g32};
    cudaError_t e = launchers[tg_lanes_index(P.lanes)](a);
    g_launches++;
    if (e != cudaSuccess) return tg_fail(100 + (int)e, "tg_sens_kernel launch", e);
    return 0;
}

// ---------------------------------------------------------------------------
// the reference's 24 symbols: single-problem launches (one warp)
// ---------------------------------------------------------------------------
enum { LG_TURN = 0, LG_MINV, LG_OBST, LG_INTERVALS, LG_BEZ };

// MDM min-norm point of the hull of 3 points (CC/src/MDMAlgorithmClass.cpp:11-71), one thread
template <int D>
__device__ double tg_mdm_min_norm3(const double *pts /* pts[c*3+i] */, int max_iterations, double tolerance)
{
    const int npts = 3;
    double p[3] = {1, 0, 0}, cur[D];
    int supp[3] = {0, 0, 0}, nsupp = 1, iterations = 0;
    double delta_p = 1.0;
    for (int c = 0; c < D; c++) cur[c] = pts[c * npts];
    while (delta_p > 0.000001 && iterations < max_iterations && nsupp > 0) {
        int max_index = supp[0], min_index = 0;
        double best = DBL_MIN;     // the reference starts from numeric_limits<double>::min()
        for (int i = 0; i < nsupp; i++) {
            double s = 0;
            for (int c = 0; c < D; c++) s += pts[c * npts + supp[i]] * cur[c];
            if (s > best) { best = s; max_index = supp[i]; }
        }
        double lo = DBL_MAX;
        for (int i = 0; i < npts; i++) {
            double s = 0;
            for (int c = 0; c < D; c++) s += pts[c * npts + i] * cur[c];
            if (s < lo) { lo = s; min_index = i; }
        }
        double diff[D], dn2 = 0;
        delta_p = 0;
        for (int c = 0; c < D; c++) {
            diff[c] = pts[c * npts + max_index] - pts[c * npts + min_index];
            delta_p += diff[c] * cur[c];
            dn2 += diff[c] * diff[c];
        }
        if (delta_p > tolerance) {
            const double dn = sqrt(dn2);
            double t = delta_p / (p[max_index] * dn * dn);
            if (t >= 1) t = 1.0;
            for (int c = 0; c < D; c++) cur[c] -= t * p[max_index] * diff[c];
            const double t1 = t * p[max_index], t2 = 1 - t;
            p[min_index] += t1;
            p[max_index] *= t2;
            nsupp = 0;
            for (int i = 0; i < npts; i++)
                if (p[i] > tolerance) supp[nsupp++] = i;
            iterations++;
        }
    }
    double s = 0;
    for (int c = 0; c < D; c++) s += cur[c] * cur[c];
    return sqrt(s);
}

template <int D>
__global__ void tg_legacy_kernel(int what, const double *pts, int N, double alpha, int kind, const double *centers,
                                 const double *radii, int K, double *out)
{
    extern __shared__ double sx[];
    const int lane = threadIdx.x;
    for (int i = lane; i < D * N; i += 32) sx[i] = pts[i];
    __syncwarp();
    const int nint = N - 3;
    if (what == LG_TURN) {
        // CC/src/CrossTermBounds.cpp:13-61
        double best = 0; int jb = 0x7fffffff;
        for (int j = lane; j < nint; j += 32) {
            TgInterval<D> I;
            tg_load_interval<D>(sx, N, j, I);
            const double b = tg_interval_turn_bound<D>(I, alpha, kind, nullptr);
            if (b > best) { best = b; jb = j; }
        }
        tg_wargmax(best, jb);
        if (lane == 0) out[0] = best;
    } else if (what == LG_MINV) {
        // CC/src/DerivativeBounds.cpp:12-27
        double best = DBL_MAX; int jb = 0x7fffffff;
        for (int j = lane; j < nint; j += 32) {
            TgInterval<D> I; double v, t;
            tg_load_interval<D>(sx, N, j, I);
            tg_min_velocity<D>(I, alpha, v, t);
            if (v < best) { best = v; jb = j; }
        }
        tg_wargmin(best, jb);
        if (lane == 0) out[0] = best;
    } else if (what == LG_OBST) {
        // CC/src/SphereCollisionEvaluator.cpp:13-45: one lane per sphere
        for (int i = lane; i < K; i += 32) {
            double ctr[D], best = DBL_MAX;
            for (int c = 0; c < D; c++) ctr[c] = centers[c * K + i];
            for (int j = 0; j < nint; j++) {
                const double dist = tg_hull_distance<D>(sx, N, j, ctr, radii[i], nullptr);
                if (best > dist) best = dist;
            }
            out[i] = best;
        }
    } else if (what == LG_INTERVALS) {
        // CC/src/SphereCollisionEvaluator.cpp:70-86: one lane per interval, sphere = (centers[0..D), radii[0])
        double ctr[D];
        for (int c = 0; c < D; c++) ctr[c] = centers[c];
        for (int j = lane; j < nint; j += 32) out[j] = tg_hull_distance<D>(sx, N, j, ctr, radii[0], nullptr);
    } else {
        // CC/src/ControlPointDerivativeBounds.cpp:13-46: N Bezier velocity points, triples at stride 2
        const int nseg = (N - 1) / 2;
        double best = DBL_MAX; int ib = 0x7fffffff;
        for (int i = lane; i < nseg; i += 32) {
            double tri[D * 3];
            for (int c = 0; c < D; c++)
                for (int l = 0; l < 3; l++) tri[c * 3 + l] = sx[c * N + 2 * i + l];
            const double v = tg_mdm_min_norm3<D>(tri, 500, 0.000001);
            if (v < best) { best = v; ib = i; }
        }
        tg_wargmin(best, ib);
        if (lane == 0) out[0] = best;
    }
}

// Result arrays: the reference returns a fresh `new double[]` from every array-returning call and never frees it
// (CC/src/ObstacleConstraints.cpp; its ctypes wrappers view it zero-copy through an ndpointer restype,
// CF/obstacle_constraints.py:53-79).  Here every call also gets a buffer of its own, so an array returned earlier is
// not overwritten by the next call; instead of leaking all of them, a handle keeps the last TG_LEGACY_RING buffers
// alive and frees the oldest (documented in INTEGRATION.md section 2).
#define TG_LEGACY_RING 64
struct LegacyHandle {
    int D;
    std::mutex mu;
    DevBuf din, dout;
    int dev = -1;
    double *ring[TG_LEGACY_RING] = {nullptr};
    unsigned long long calls = 0;
};

static void *tg_new_handle(int D)
{
    LegacyHandle *h = new LegacyHandle();
    h->D = D;
    return h;
}

// runs one legacy query; returns pointer to nout doubles owned by the handle (NaN-filled on failure)
static double *tg_legacy_run(void *obj, int D, int what, const double *pts, int N, double alpha, int kind,
                             const double *centers, const double *radii, int K, int nout)
{
    static LegacyHandle fallback[2];
    LegacyHandle *h = obj ? (LegacyHandle *)obj : &fallback[D - 2];
    std::lock_guard<std::mutex> lock(h->mu);
    double *&slot = h->ring[h->calls++ % TG_LEGACY_RING];
    delete[] slot;
    slot = new double[(size_t)nout + 1];
    double *res = slot;
    for (int i = 0; i < nout; i++) res[i] = NAN;
    if (tg_device_check()) { fprintf(stderr, "libTrajectoryConstraints (B200): %s\n", g_err); return res; }
    if (N < 4 && what != LG_BEZ) { fprintf(stderr, "libTrajectoryConstraints (B200): need at least 4 control points\n"); return res; }
    const int nc = (what == LG_INTERVALS) ? D : D * K;
    const int nr = (what == LG_INTERVALS) ? 1 : K;
    const size_t nin = (size_t)D * N + nc + nr;
    int dev = 0;
    cudaGetDevice(&dev);
    if (h->dev != dev) { h->din = DevBuf(); h->dout = DevBuf(); h->dev = dev; }     // buffers belong to the device they were made on
    if (h->din.ensure((nin + 1) * sizeof(double)) || h->dout.ensure(((size_t)nout + 1) * sizeof(double))) {
        fprintf(stderr, "libTrajectoryConstraints (B200): %s\n", g_err);
        return res;
    }
    double *dpts = (double *)h->din.p, *dctr = dpts + (size_t)D * N, *drad = dctr + nc;
    cudaMemcpyAsync(dpts, pts, sizeof(double) * D * N, cudaMemcpyHostToDevice, 0);
    if (centers && nc) cudaMemcpyAsync(dctr, centers, sizeof(double) * nc, cudaMemcpyHostToDevice, 0);
    if (radii && nr) cudaMemcpyAsync(drad, radii, sizeof(double) * nr, cudaMemcpyHostToDevice, 0);
    const size_t smem = sizeof(double) * ((size_t)D * N + 1);
    if (D == 2) tg_legacy_kernel<2><<<1, 32, smem, 0>>>(what, dpts, N, alpha, kind, dctr, drad, K, (double *)h->dout.p);
    else tg_legacy_kernel<3><<<1, 32, smem, 0>>>(what, dpts, N, alpha, kind, dctr, drad, K, (double *)h->dout.p);
    g_launches++;
    cudaError_t e = cudaMemcpy(res, h->dout.p, sizeof(double) * nout, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
        fprintf(stderr, "libTrajectoryConstraints (B200): %s\n", cudaGetErrorString(e));
        for (int i = 0; i < nout; i++) res[i] = NAN;
    }
    return res;
}

#define TG_DEFINE_LEGACY(D)                                                                                            \
    extern "C" void *CrossTermBounds_##D(void) { return tg_new_handle(D); }                                            \
    extern "C" double get_spline_curvature_bound_##D(void *o, double p[], int N)                                       \
    { return tg_legacy_run(o, D, LG_TURN, p, N, 1.0, TG_TURN_CURVATURE, 0, 0, 0, 1)[0]; }                              \
    extern "C" double get_spline_angular_rate_bound_##D(void *o, double p[], int N, double a)                          \
    { return tg_legacy_run(o, D, LG_TURN, p, N, a, TG_TURN_ANGULAR_RATE, 0, 0, 0, 1)[0]; }                             \
    extern "C" double get_spline_centripetal_acceleration_bound_##D(void *o, double p[], int N, double a)              \
    { return tg_legacy_run(o, D, LG_TURN, p, N, a, TG_TURN_CENTRIPETAL, 0, 0, 0, 1)[0]; }                              \
    extern "C" void *DerivativeBounds_##D(void) { return tg_new_handle(D); }                                           \
    extern "C" double find_min_velocity_of_spline_##D(void *o, double p[], int N, double a)                            \
    { return tg_legacy_run(o, D, LG_MINV, p, N, a, 0, 0, 0, 0, 1)[0]; }                                                \
    extern "C" void *ObstacleConstraints_##D(void) { return tg_new_handle(D); }                                        \
    extern "C" double *getObstaclesConstraintsForSpline_##D(void *o, double c[], double r[], int K, double p[], int N) \
    { return tg_legacy_run(o, D, LG_OBST, p, N, 1.0, 0, c, r, K, K > 0 ? K : 1); }                                     \
    extern "C" double *getObstacleConstraintsForIntervals_##D(void *o, double p[], int N, double r, double c[])        \
    { return tg_legacy_run(o, D, LG_INTERVALS, p, N, 1.0, 0, c, &r, 1, N - 3 > 0 ? N - 3 : 1); }                       \
    extern "C" double getObstacleConstraintForSpline_##D(void *o, double p[], int N, double r, double c[])             \
    {                                                                                                                  \
        double *a = tg_legacy_run(o, D, LG_INTERVALS, p, N, 1.0, 0, c, &r, 1, N - 3 > 0 ? N - 3 : 1);                  \
        double b = DBL_MAX;                                                                                            \
        for (int j = 0; j < N - 3; j++) { if (a[j] != a[j]) return a[j]; if (b > a[j]) b = a[j]; }                     \
        return b;                                                                                                      \
    }                                                                                                                  \
    extern "C" void *ControlPointDerivativeBounds_##D(void) { return tg_new_handle(D); }                               \
    extern "C" double find_min_velocity_of_bez_vel_cont_pts_##D(void *o, double p[], int n)                            \
    { return tg_legacy_run(o, D, LG_BEZ, p, n, 1.0, 0, 0, 0, 0, 1)[0]; }

TG_DEFINE_LEGACY(2)
TG_DEFINE_LEGACY(3)
