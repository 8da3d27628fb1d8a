// Parameter sensitivities of a converged solve by the implicit-function theorem on its KKT system: one adjoint solve per
// problem (tg_sens_kernel, tg_kernels_sens.inc; the host build under tests/hostsim; DESIGN.md §4 *Sensitivities*).
//
// For one problem with status 0 at x* with multipliers lam, and upstream gradients x_bar[n] and f_bar of a scalar loss,
// par_bar = d(loss)/d(par).  With the polish's definitions (tg_polish.h): F the free variables, W every equality row and
// the inequality rows with lam_j > 0, A_W the Jacobian of the W rows over F:
//   1. g_bar = x_bar + f_bar grad f(x*)            (the objective does not read par: df*/dp = grad f . dx*/dp)
//   2. Householder QR A_W' = [Y Z] [R; 0]; least-squares multipliers lam_W = R^-1 Y' g_F
//   3. H = d2L/dx2 over F with lam_W (tg_polish_hessian: central differences of the analytic gradL)
//   4. adjoint of [H A_W'; A_W 0]:  u = Z (Z'HZ)^-1 Z' g_bar_F  (unshifted Cholesky: a shifted Hessian would differentiate
//      another problem),  w = R^-1 Y' (g_bar_F - H u)
//   5. psi(p) = sum_{j in W} lam_j (grad_x c_j(x*, p) . u) - w_j c_j(x*, p);  par_bar = d psi / dp by central differences
//      over every entry k of the row, step h_k = eps^(1/3) max(1, |p_k|), divided by (p_k + h) - (p_k - h).  grad_x c
//      includes the LINEAR rows: the corridor rows' coefficients and the moving-target end rows' alpha column depend on
//      par.  The entry is perturbed in the problem's scratch copy of par and restored from the input bit for bit.
// Statuses (first match wins): skipped (status != 0), degenerate (|W| > |F| or |R_kk| < 1e-12 max|R|), indefinite (no
// unshifted Cholesky of Z'HZ), nonfinite -- these rows get zeros; inexact (stationarity with the given lam and analytic
// derivatives > tol max(1, max|g|), or a least-squares lam_j < 0 on an inequality row of W) and nonstrict (an
// inequality row outside W with c_j <= 1e-8, or one in W with lam_j <= 1e-8 max(1, max|lam_W|): the derivative holds W
// fixed and is one-sided) -- these rows are computed and returned.
// Cost: 1 + 2 |F| evaluations with derivatives for H, 2 P for psi.  Every sum runs in a fixed order on one lane and
// every lane-parallel loop writes entries of its own: results do not depend on placement, instantiation, lane count or
// batch position.
#ifndef TG_SENS_H
#define TG_SENS_H

#include "tg_polish.h"

enum { TG_SENS_OK = 0, TG_SENS_NONSTRICT, TG_SENS_INEXACT, TG_SENS_DEGENERATE, TG_SENS_SKIPPED, TG_SENS_NONFINITE,
       TG_SENS_INDEFINITE };

// Per-problem scratch: the polish's (tg_polish_carve), then u[n] (the adjoint over F) and w[m + 1] (row order)
struct TgSensWs {
    TgPolishWs P;
    double *u, *w;
};

TG_HD size_t tg_sens_carve(const TgLayout &L, double *base, TgSensWs *S)
{
    TgPolishWs P;
    size_t o = tg_polish_carve(L, base, &P);
    double *u = base + o;
    o += (size_t)L.n; o += o & 1;
    double *w = base + o;
    o += (size_t)L.m + 1; o += o & 1;
    if (S) { S->P = P; S->u = u; S->w = w; }
    return o;
}
TG_HD size_t tg_sens_group_doubles(const TgLayout &L) { return tg_sens_carve(L, 0, 0); }

// psi at P.par with entry k set to v (restored by the caller): c and EVERY Jacobian row (linear ones included, at the
// perturbed par) at x*, then sum over W in row order of lam_j (J_j . u) - w_j c_j; every lane returns the same value
template <int D>
TG_FN double tg_sens_psi(const TgLayout &L, const int *sp, const TgSensWs &S, int nF, int nW, int k, double v)
{
    const TgPolishWs &P = S.P;
    const int lane = TG_LANE(), n = L.n;
    if (lane == 0) P.par[k] = v;
    TG_SYNC();
    const TgJac sink = {P.J, n, 1, 0};
    tg_constraints_d<D>(L, sp, P.par, P.x, P.ct, &sink, P.scratch);
    tg_linear_jacobian_d<D>(L, sp, P.par, sink);
    #pragma unroll 1
    for (int q = lane; q < nW; q += TG_NL) {
        const int j = P.wrow[q];
        const double *row = P.J + (size_t)j * n;
        double d = 0;
        #pragma unroll 1
        for (int a = 0; a < nF; a++) d += row[P.fr[a]] * S.u[a];
        P.tmp[q] = P.lam[j] * d - S.w[j] * P.ct[j];
    }
    TG_SYNC();
    double psi = 0;
    #pragma unroll 1
    for (int q = 0; q < nW; q++) psi += P.tmp[q];
    TG_SYNC();
    return psi;
}

// One problem (see the top of the file).  sp / par: descriptor and parameter row; x[n], status, lam[m]: the solve's
// outputs; x_bar[n], f_bar: upstream gradients; par_bar[P] and *sstatus: outputs.
template <int D>
TG_FN void tg_sens_problem(const TgLayout &L, const int *sp, const double *par, double *ws, const double *xin, int status,
                           const double *lamin, const double *xbar, double fbar, double *pbar, int *sstatus, double tol)
{
    const int lane = TG_LANE(), n = L.n, m = L.m, meq = L.meq, np = L.P;
    int code = TG_SENS_OK;
    TgSensWs S;
    tg_sens_carve(L, ws, &S);
    const TgPolishWs &P = S.P;
    if (status != 0) { code = TG_SENS_SKIPPED; goto zero; }
    {
        #pragma unroll 1
        for (int i = lane; i < np; i += TG_NL) P.par[i] = par[i];
        #pragma unroll 1
        for (int i = lane; i < n; i += TG_NL) {
            tg_polish_bounds(L, i, P.xl[i], P.xu[i]);
            P.x[i] = P.xt[i] = xin[i];
        }
        #pragma unroll 1
        for (int j = lane; j < m; j += TG_NL) { P.lam[j] = lamin[j]; P.drop[j] = 0; }
        #pragma unroll 1
        for (size_t q = lane; q < (size_t)m * n; q += TG_NL) P.J[q] = 0;
        TG_SYNC();
        {
            const TgJac sink = {P.J, n, 1, 0};
            tg_linear_jacobian_d<D>(L, sp, P.par, sink);
        }
        tg_polish_eval<D>(L, sp, P);
        double kkt[4], gmax;
        tg_polish_kkt(L, P, P.lam, kkt, &gmax);
        int inexact = !(kkt[0] <= tol * fmax(1.0, gmax));
        int nF, nW;
        tg_polish_sets(L, P, &nF, &nW);
        if (nW > nF || tg_polish_qr(L, P, nF, nW)) { code = TG_SENS_DEGENERATE; goto zero; }
        // least-squares multipliers lam_W = R^-1 (Q'g_F)_y, into P.lam (zeros outside W): the Hessian and psi use them
        if (lane == 0) {
            for (int a = 0; a < nF; a++) P.gq[a] = P.g[P.fr[a]];
            for (int k = 0; k < nW; k++) tg_polish_reflect(P, nF, k, P.gq);
            for (int k = 0; k < nW; k++) P.tmp[k] = P.gq[k];
            tg_polish_rsolve(P, nF, nW, P.tmp);
            for (int j = 0; j < m; j++) P.lam[j] = 0;
            for (int k = 0; k < nW; k++) P.lam[P.wrow[k]] = P.tmp[k];
        }
        TG_SYNC();
        // strictness (c at x*, P.c) and the signs of lam_W; W is sorted, so a walk finds the inequality rows outside it
        double lwmax = 0;
        #pragma unroll 1
        for (int k = 0; k < nW; k++) lwmax = tg_kkt_fold(lwmax, fabs(P.lam[P.wrow[k]]));
        int nonstrict = 0;
        #pragma unroll 1
        for (int j = meq, q = 0; j < m; j++) {
            while (q < nW && P.wrow[q] < j) q++;
            if (q < nW && P.wrow[q] == j) {
                inexact |= P.lam[j] < 0;
                nonstrict |= P.lam[j] <= 1e-8 * fmax(1.0, lwmax);
            } else {
                nonstrict |= P.c[j] <= 1e-8;
            }
        }
        // H with lam_W, C = Q'HQ, unshifted Cholesky of Z'HZ
        tg_polish_hessian<D>(L, sp, P, nF);
        tg_polish_reduce(P, nF, nW);
        const int nz = nF - nW;
        if (nz > 0 && !tg_polish_chol(P, nF, nW, 0.0)) { code = TG_SENS_INDEFINITE; goto zero; }
        // adjoint: gq = Q'g_bar_F, t = (Z'HZ)^-1 gq_z in pq[nW..], pq[..nW) = 0; w_W = R^-1 (gq_y - C_yz t); u_F = Q pq
        if (lane == 0) {
            for (int a = 0; a < nF; a++) P.gq[a] = xbar[P.fr[a]] + fbar * P.g[P.fr[a]];
            for (int k = 0; k < nW; k++) tg_polish_reflect(P, nF, k, P.gq);
            for (int a = 0; a < nz; a++) P.tmp[a] = P.gq[nW + a];
            tg_polish_chol_solve(P, nz, P.tmp);
            for (int k = 0; k < nW; k++) P.pq[k] = 0;
            for (int a = 0; a < nz; a++) P.pq[nW + a] = P.tmp[a];
        }
        TG_SYNC();
        #pragma unroll 1
        for (int k = lane; k < nW; k += TG_NL) {
            const double *row = P.C + (size_t)k * nF;
            double s = P.gq[k];
            #pragma unroll 1
            for (int b = nW; b < nF; b++) s -= row[b] * P.pq[b];
            P.tmp[k] = s;
        }
        TG_SYNC();
        if (lane == 0) {
            tg_polish_rsolve(P, nF, nW, P.tmp);
            for (int j = 0; j < m; j++) S.w[j] = 0;
            for (int k = 0; k < nW; k++) S.w[P.wrow[k]] = P.tmp[k];
            for (int k = nW - 1; k >= 0; k--) tg_polish_reflect(P, nF, k, P.pq);
            for (int a = 0; a < nF; a++) S.u[a] = P.pq[a];
        }
        TG_SYNC();
        // par_bar by central differences of psi, one entry at a time
        int bad = 0;
        #pragma unroll 1
        for (int k = 0; k < np; k++) {
            const double pk = par[k], h = TG_POLISH_H_REL * fmax(1.0, fabs(pk)), pp = pk + h, pm = pk - h;
            const double psip = tg_sens_psi<D>(L, sp, S, nF, nW, k, pp);
            const double psim = tg_sens_psi<D>(L, sp, S, nF, nW, k, pm);
            if (lane == 0) P.par[k] = pk;
            const double v = (psip - psim) / (pp - pm);
            bad |= !tg_finite(v);
            if (lane == 0) pbar[k] = v;
        }
        TG_SYNC();
        if (bad) { code = TG_SENS_NONFINITE; goto zero; }
        if (lane == 0) *sstatus = inexact ? TG_SENS_INEXACT : nonstrict ? TG_SENS_NONSTRICT : TG_SENS_OK;
        return;
    }
zero:
    #pragma unroll 1
    for (int k = lane; k < np; k += TG_NL) pbar[k] = 0;
    if (lane == 0) *sstatus = code;
    TG_SYNC();
}

#endif  // TG_SENS_H
