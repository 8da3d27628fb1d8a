// M2, fused form: one persistent kernel, each warp runs both SQP stages of a problem until it is done.  Kept for
// comparison with the lock-step stage kernels (profiles/README.md: it is instruction-cache bound); the QP-stage
// functions stay out of line here.
#define TG_GS 32
#define TG_SQP_NOINLINE
#include "tg_sqp.h"
#include "tg_shape.h"

// ---------------------------------------------------------------------------
// fused form: persistent CTAs, each warp pulls problem indices from an atomic queue and runs both stages
// until its problem is done (kept for comparison; see profiles/README.md)
// ---------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(128, 4)
tg_solve_kernel(const TgShape S, int B, const double *__restrict__ par, double *__restrict__ x, double *__restrict__ fout,
                int *__restrict__ status, int *__restrict__ nit, int *__restrict__ violation, double *__restrict__ lam,
                double *__restrict__ kkt, int maxiter, double ftol, int flags, double *gws, size_t ws_doubles,
                int warps_per_cta, int *queue)
{
    extern __shared__ double smem[];
    const TgLayout &L = S.L;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // per-warp slice: parameters + (shared-memory workspace | pointer into the global one)
    double *spar = smem + (size_t)warp * (L.P + (gws ? 0 : ws_doubles) + 2);
    double *ws = gws ? gws + ((size_t)blockIdx.x * warps_per_cta + warp) * ws_doubles : spar + L.P + 1;
    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(queue, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= B) break;
        for (int i = lane; i < L.P; i += 32) spar[i] = par[(size_t)b * L.P + i];
        __syncwarp();
        TgSqpResult res;
        tg_sqp_solve<D>(L, S.sp, spar, x + (size_t)b * L.n, ws, maxiter, ftol, flags, &res, nullptr, 0);
        res.status = __shfl_sync(0xffffffffu, res.status, 0);
        int viol = 0;
        TgSqpWs W;
        tg_sqp_carve(L, ws, &W);
        if (res.status != 0) viol = tg_last_block_violation(L, W.c);
        // (the solve's scratch is free now: its vector u, n + 1 doubles, serves tg_sqp_kkt)
        if (lam || kkt) tg_sqp_kkt(L, W, lam ? lam + (size_t)b * L.m : nullptr, kkt ? kkt + (size_t)b * 4 : nullptr, W.u);
        if (lane == 0) {
            if (status) status[b] = res.status;
            if (nit) nit[b] = res.nit;
            if (fout) fout[b] = res.f;
            if (violation) violation[b] = viol;
        }
        __syncwarp();
    }
}

// grid and workspace of the fused kernel: a shared-memory workspace per warp when at least 8 warps fit on an SM, else
// a global one (per resident warp) in the solve workspace
struct TgFusedPlan {
    int warps_per_cta, ctas, use_global;
    size_t ws_doubles, smem_bytes, global_bytes;
};

static TgFusedPlan tg_fused_plan(const TgShape &S, int B, int sm_count, int smem_optin)
{
    TgFusedPlan P;
    const size_t budget = (size_t)smem_optin - 1024;
    const size_t sm_total = 227 * 1024;
    P.ws_doubles = tg_sqp_workspace_doubles(S.L);
    const size_t per_warp_shared = (S.L.P + P.ws_doubles + 2) * sizeof(double);
    if (per_warp_shared * 8 <= sm_total) {
        P.use_global = 0;
        P.warps_per_cta = 4;
        while (per_warp_shared * P.warps_per_cta > budget) P.warps_per_cta >>= 1;
        P.smem_bytes = per_warp_shared * P.warps_per_cta;
        int per_sm = (int)(sm_total / (P.smem_bytes + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm * P.warps_per_cta > 32) per_sm = 32 / P.warps_per_cta;
        P.ctas = sm_count * per_sm;
    } else {
        P.use_global = 1;
        P.warps_per_cta = 4;
        P.smem_bytes = (size_t)P.warps_per_cta * (S.L.P + 2) * sizeof(double);
        P.ctas = sm_count * 4;
    }
    const int need = (B + P.warps_per_cta - 1) / P.warps_per_cta;
    if (P.ctas > need) P.ctas = need > 0 ? need : 1;
    P.global_bytes = P.use_global ? (size_t)P.ctas * P.warps_per_cta * P.ws_doubles * sizeof(double) : 0;
    return P;
}

size_t tg_fused_workspace_bytes(const TgShape &S, int B, int sm_count, int smem_optin)
{
    return tg_fused_plan(S, B, sm_count, smem_optin).global_bytes;
}

cudaError_t tg_launch_fused_g32(const TgShape &S, int B, const double *par, double *x, double *f, int *status, int *nit,
                                int *violation, double *lam, double *kkt, int maxiter, double ftol, int flags, void *gws,
                                int *queue, int sm_count, int smem_optin, cudaStream_t st)
{
    const TgFusedPlan P = tg_fused_plan(S, B, sm_count, smem_optin);
    double *ws = P.use_global ? (double *)gws : nullptr;
    cudaError_t e;
    if (S.L.d == 2) {
        if ((e = tg_allow_shared_memory(tg_solve_kernel<2>))) return e;
        tg_solve_kernel<2><<<P.ctas, P.warps_per_cta * 32, P.smem_bytes, st>>>(S, B, par, x, f, status, nit, violation, lam, kkt, maxiter,
                                                                                ftol, flags, ws, P.ws_doubles, P.warps_per_cta, queue);
    } else {
        if ((e = tg_allow_shared_memory(tg_solve_kernel<3>))) return e;
        tg_solve_kernel<3><<<P.ctas, P.warps_per_cta * 32, P.smem_bytes, st>>>(S, B, par, x, f, status, nit, violation, lam, kkt, maxiter,
                                                                                ftol, flags, ws, P.ws_doubles, P.warps_per_cta, queue);
    }
    return cudaGetLastError();
}
