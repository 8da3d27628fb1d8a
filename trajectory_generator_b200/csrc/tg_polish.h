// Post-solve polish of a converged problem: safeguarded Newton steps on the KKT system of SLSQP's final active set with
// an exact Lagrangian Hessian (tg_polish_kernel, tg_kernels_polish.inc; the host build under tests/hostsim).
// The parameter sensitivities (tg_sens.h) call its working set, Hessian, QR and Cholesky functions as well.
//
// SLSQP stops when |f - f0| or the step falls below its tolerance.  A badly conditioned BFGS factor makes the step tiny
// while the Lagrangian gradient is still large, so a status-0 point is feasible and complementary but often not
// stationary (DESIGN.md §4).  For one problem with status 0, given the solve's x and multipliers lam:
//   working set W   every equality row, the inequality rows with lam_j > 0 (the last QP's active rows), and the
//                   variables at a bound (x_i == xl_i or x_i == xu_i, the test tg_sqp_kkt makes) held fixed;
//                   |W| > free variables or a rank-deficient A_W (|R_kk| < 1e-12 max|R|): `degenerate`
//   Hessian         H = d2L/dx2 (x, lam) by central differences of the ANALYTIC gradL = g - J' lam over the free
//                   variables (the linear rows drop out), step eps^(1/3) max(1, |x_i|), one-sided at a bound;
//                   symmetrised.  2 n_free + 1 evaluations per Newton step -- analytic even after an fd-mode solve.
//   step            null-space method: Householder QR of A_W' over the free variables, range-space part from c_W,
//                   Cholesky of Z'HZ (+ delta I, delta = 0, 1e-8 max|H|, x100, at most 4 tries), least-squares
//                   multipliers lam_W from the range-space equations.  An inequality row of W with lam_j < 0 is
//                   dropped (the most negative one) and the step recomputed: that counts as one iteration.
//   globalisation   backtracking alpha in {1, 1/2, 1/4, 1/8} on the l1 merit f + rho sum(violations),
//                   rho = 1 + 2 max|lam_in|, the trial x clipped to the bounds.  Stop when the stationarity is
//                   <= tol max(1, max|g|) or after maxiter iterations.
//   final guard     the polished row replaces the input only if every value is finite, the maximum violation is
//                   <= max(v_in, 1e-8), merit_out <= merit_in, stationarity_out < stationarity_in (both with the
//                   analytic derivatives) and the dual infeasibility is <= 1e-8 max(1, max|lam|).  Otherwise x, f,
//                   lam, kkt and violation stay bit for bit as they were.
// A replaced row gets x, f, lam (lam_W in row order, zeros elsewhere), kkt[4] at the new x with the definitions of
// tg_sqp_kkt (restated here over a dense Jacobian) and the reference's violation flag (tg_last_block_violation).
// Every sum runs in a fixed order on one lane, and every lane-parallel loop writes entries of its own: the results do
// not depend on the placement, the instantiation or the batch position.  (The objective's value comes from
// tg_objective, whose sum is folded across the lanes of the group: the host build's single lane may differ from the
// device in the last bits of f.)
#ifndef TG_POLISH_H
#define TG_POLISH_H

#include "tg_sqp.h"

enum { TG_POLISH_POLISHED = 0, TG_POLISH_IMPROVED, TG_POLISH_REJECTED, TG_POLISH_DEGENERATE, TG_POLISH_SKIPPED,
       TG_POLISH_NONFINITE };

#define TG_POLISH_H_REL 6.0554544523933395e-06      // cbrt(DBL_EPSILON): central-difference step relative to max(1, |x|)

// Per-problem scratch, in doubles: [par | x xt xl xu g gp gq pq tmp beta rdiag | c ct lam lamw | J (m x n) |
// Jp (m_nl x n) | H C F AT (n x n each) | ints: free[n] wrow[m] drop[m] | evaluators' scratch]
struct TgPolishWs {
    double *par, *x, *xt, *xl, *xu, *g, *gp, *gq, *pq, *tmp, *beta, *rdiag, *c, *ct, *lam, *lamw, *J, *Jp, *H, *C, *F, *AT;
    int *fr, *wrow, *drop;
    double *scratch;
};

TG_HD size_t tg_polish_carve(const TgLayout &L, double *base, TgPolishWs *P)
{
    const size_t n = (size_t)L.n, m = (size_t)L.m;
    size_t o = 0;
    TgPolishWs w;
#define TG_PTAKE(field, count) w.field = base + o; o += (size_t)(count); o += o & 1
    TG_PTAKE(par, L.P);
    TG_PTAKE(x, n); TG_PTAKE(xt, n); TG_PTAKE(xl, n); TG_PTAKE(xu, n); TG_PTAKE(g, n); TG_PTAKE(gp, n);
    TG_PTAKE(gq, n); TG_PTAKE(pq, n); TG_PTAKE(tmp, n); TG_PTAKE(beta, n); TG_PTAKE(rdiag, n);
    TG_PTAKE(c, m + 1); TG_PTAKE(ct, m + 1); TG_PTAKE(lam, m + 1); TG_PTAKE(lamw, m + 1);
    TG_PTAKE(J, m * n); TG_PTAKE(Jp, (size_t)L.m_nl * n);
    TG_PTAKE(H, n * n); TG_PTAKE(C, n * n); TG_PTAKE(F, n * n); TG_PTAKE(AT, n * n);
    w.fr = (int *)(base + o); w.wrow = w.fr + n; w.drop = w.wrow + m;
    o += (n + 2 * m) / 2 + 1; o += o & 1;
    TG_PTAKE(scratch, tg_scratch_doubles(L));
#undef TG_PTAKE
    if (P) *P = w;
    return o;
}
TG_HD size_t tg_polish_group_doubles(const TgLayout &L) { return tg_polish_carve(L, 0, 0); }

// bounds of the variables: tg_sqp_begin's (TG/objectives/objective_variables.py:50-61)
TG_HD void tg_polish_bounds(const TgLayout &L, int i, double &lo, double &hi)
{
    lo = -INFINITY; hi = INFINITY;
    if (i >= L.ia && i < L.it0) lo = 10e-8;
    if (i >= L.it0 && i < L.n) { lo = 0; hi = L.N - 3; }
}

// true maximum violation (multi-start's fold: |c| equality rows, max(0, -c) inequality rows, NaN -> +inf); every lane
TG_HD double tg_polish_maxviol(const TgLayout &L, const double *c)
{
    double v = 0;
    #pragma unroll 1
    for (int j = TG_LANE(); j < L.m; j += TG_NL) v = tg_kkt_fold(v, j < L.meq ? fabs(c[j]) : fmax(-c[j], 0.0));
    int k = 0;
    tg_wargmax(v, k);
    return v;
}

// l1 merit f + rho sum(violations), summed in row order; every lane
TG_HD double tg_polish_merit(const TgLayout &L, double f, const double *c, double rho)
{
    double h = 0;
    #pragma unroll 1
    for (int j = 0; j < L.m; j++) h += j < L.meq ? fabs(c[j]) : fmax(-c[j], 0.0);
    return f + rho * h;
}

// kkt[4] at x from g, c, the dense Jacobian J (all m rows) and lam: tg_sqp_kkt's definitions; returns max|g| in *gmax
TG_HD void tg_polish_kkt(const TgLayout &L, const TgPolishWs &P, const double *lam, double *kkt, double *gmax)
{
    const int n = L.n, m = L.m;
    double st = 0, gm = 0;
    #pragma unroll 1
    for (int i = TG_LANE(); i < n; i += TG_NL) {
        double h = P.g[i];
        #pragma unroll 1
        for (int r = 0; r < m; r++)
            if (lam[r] != 0) h -= P.J[(size_t)r * n + i] * lam[r];
        const double pi = P.x[i] == P.xl[i] ? fmin(h, 0.0) : P.x[i] == P.xu[i] ? fmax(h, 0.0) : h;
        st = tg_kkt_fold(st, fabs(pi));
        gm = tg_kkt_fold(gm, fabs(P.g[i]));
    }
    double inf = 0, dinf = 0, comp = 0;
    #pragma unroll 1
    for (int j = TG_LANE(); j < m; j += TG_NL) {
        const double cj = P.c[j];
        if (j < L.meq) { inf = tg_kkt_fold(inf, fabs(cj)); continue; }
        inf = tg_kkt_fold(inf, -cj);
        dinf = tg_kkt_fold(dinf, -lam[j]);
        comp = tg_kkt_fold(comp, fabs(lam[j] * cj));
    }
    int k0 = 0;
    tg_wargmax(st, k0); tg_wargmax(gm, k0); tg_wargmax(inf, k0); tg_wargmax(dinf, k0); tg_wargmax(comp, k0);
    kkt[0] = st; kkt[1] = inf; kkt[2] = dinf; kkt[3] = comp;
    *gmax = gm;
}

// f, g, c and the nonlinear rows of the dense Jacobian at P.x (the linear rows of P.J are set once)
template <int D>
TG_FN double tg_polish_eval(const TgLayout &L, const int *sp, const TgPolishWs &P)
{
    const double f = tg_objective(L, sp, P.x, P.g);
    TgJac sink = {P.J, L.n, 1, 0};
    tg_constraints_d<D>(L, sp, P.par, P.x, P.c, &sink, P.scratch);
    TG_SYNC();
    return f;
}

// gradL over the free variables at P.xt, the linear rows left out: gp[a] = g_F(a) - sum_nonlinear Jp' lam
template <int D>
TG_FN void tg_polish_gradl(const TgLayout &L, const int *sp, const TgPolishWs &P, int nF)
{
    const int n = L.n;
    tg_objective(L, sp, P.xt, P.tmp);
    TgJac sink = {P.Jp, n, 1, 1};
    tg_constraints_d<D>(L, sp, P.par, P.xt, P.ct, &sink, P.scratch, TG_SKIP_LINEAR);
    TG_SYNC();
    #pragma unroll 1
    for (int a = TG_LANE(); a < nF; a += TG_NL) {
        const int i = P.fr[a];
        double h = P.tmp[i];
        #pragma unroll 1
        for (int r = 0; r < L.m; r++) {
            const int q = tg_nlrow(L, r);
            if (q >= 0 && P.lam[r] != 0) h -= P.Jp[(size_t)q * n + i] * P.lam[r];
        }
        P.gp[a] = h;
    }
    TG_SYNC();
}

// v = the Householder vector k (AT column k from entry k on), applied as (I - beta v v') to vec[k..nF) on lane 0
TG_HD void tg_polish_reflect(const TgPolishWs &P, int nF, int k, double *vec)
{
    const double *v = P.AT + (size_t)k * nF;
    double s = 0;
    #pragma unroll 1
    for (int a = k; a < nF; a++) s += v[a] * vec[a];
    s *= P.beta[k];
    #pragma unroll 1
    for (int a = k; a < nF; a++) vec[a] -= s * v[a];
}

// free variables (P.fr, x strictly inside its bounds) and working set (P.wrow: every equality row and the inequality
// rows with lam_j > 0 not marked in P.drop), both in index order; every lane
TG_HD void tg_polish_sets(const TgLayout &L, const TgPolishWs &P, int *nFo, int *nWo)
{
    const int lane = TG_LANE();
    int nF = 0, nW = 0;
    #pragma unroll 1
    for (int i = 0; i < L.n; i++)
        if (P.x[i] != P.xl[i] && P.x[i] != P.xu[i]) { if (lane == 0) P.fr[nF] = i; nF++; }
    #pragma unroll 1
    for (int j = 0; j < L.m; j++)
        if (j < L.meq || (P.lam[j] > 0 && !P.drop[j])) { if (lane == 0) P.wrow[nW] = j; nW++; }
    TG_SYNC();
    *nFo = nF; *nWo = nW;
}

// H (nF x nF, row-major) = d2L/dx2 over the free variables at P.x with the multipliers P.lam: column b from
// tg_polish_gradl at x +- h e_i, h = eps^(1/3) max(1, |x_i|), one-sided at a bound; symmetrised
template <int D>
TG_FN void tg_polish_hessian(const TgLayout &L, const int *sp, const TgPolishWs &P, int nF)
{
    const int lane = TG_LANE();
    #pragma unroll 1
    for (int b = 0; b < nF; b++) {
        const int i = P.fr[b];
        const double xi = P.x[i], h = TG_POLISH_H_REL * fmax(1.0, fabs(xi));
        const double xp = fmin(xi + h, P.xu[i]), xm = fmax(xi - h, P.xl[i]);
        if (lane == 0) P.xt[i] = xp;
        TG_SYNC();
        tg_polish_gradl<D>(L, sp, P, nF);
        #pragma unroll 1
        for (int a = lane; a < nF; a += TG_NL) P.H[(size_t)a * nF + b] = P.gp[a];
        if (lane == 0) P.xt[i] = xm;
        TG_SYNC();
        tg_polish_gradl<D>(L, sp, P, nF);
        #pragma unroll 1
        for (int a = lane; a < nF; a += TG_NL) P.H[(size_t)a * nF + b] = (P.H[(size_t)a * nF + b] - P.gp[a]) / (xp - xm);
        if (lane == 0) P.xt[i] = xi;
        TG_SYNC();
    }
    #pragma unroll 1
    for (int a = lane; a < nF; a += TG_NL)
        #pragma unroll 1
        for (int b = a + 1; b < nF; b++) {
            const double s = 0.5 * (P.H[(size_t)a * nF + b] + P.H[(size_t)b * nF + a]);
            P.H[(size_t)a * nF + b] = s; P.H[(size_t)b * nF + a] = s;
        }
    TG_SYNC();
}

// Householder QR of A_W' (nF x nW, column k = Jacobian row W_k over the free variables) in place in P.AT: reflector k
// is AT column k from entry k on with P.beta[k]; R_kk = rdiag[k], R_kj = AT[j][k] (j > k).  Returns 1 when A_W is
// rank-deficient (some |R_kk| < 1e-12 max|R|); every lane
TG_FN int tg_polish_qr(const TgLayout &L, const TgPolishWs &P, int nF, int nW)
{
    const int lane = TG_LANE(), n = L.n;
    #pragma unroll 1
    for (int q = lane; q < nF * nW; q += TG_NL) {
        const int k = q / nF, a = q - k * nF;
        P.AT[q] = P.J[(size_t)P.wrow[k] * n + P.fr[a]];
    }
    TG_SYNC();
    #pragma unroll 1
    for (int k = 0; k < nW; k++) {
        double *v = P.AT + (size_t)k * nF;
        double s = 0;
        #pragma unroll 1
        for (int a = k; a < nF; a++) s += v[a] * v[a];
        const double nrm = sqrt(s), vk0 = v[k];
        const double alpha = vk0 > 0 ? -nrm : nrm, vk = vk0 - alpha;
        const double beta = nrm > 0 ? -1.0 / (alpha * vk) : 0.0;
        TG_SYNC();
        if (lane == 0) { v[k] = vk; P.beta[k] = beta; P.rdiag[k] = alpha; }
        TG_SYNC();
        #pragma unroll 1
        for (int j = k + 1 + lane; j < nW; j += TG_NL) {
            double *col = P.AT + (size_t)j * nF;
            double t = 0;
            #pragma unroll 1
            for (int a = k; a < nF; a++) t += v[a] * col[a];
            t *= beta;
            #pragma unroll 1
            for (int a = k; a < nF; a++) col[a] -= t * v[a];
        }
        TG_SYNC();
    }
    double rmax = 0;
    #pragma unroll 1
    for (int q = lane; q < nW * nW; q += TG_NL) {
        const int j = q / nW, k = q - j * nW;
        if (k < j) rmax = tg_kkt_fold(rmax, fabs(P.AT[(size_t)j * nF + k]));
        else if (k == j) rmax = tg_kkt_fold(rmax, fabs(P.rdiag[k]));
    }
    int k0 = 0;
    tg_wargmax(rmax, k0);
    int rankdef = 0;
    #pragma unroll 1
    for (int k = 0; k < nW; k++) rankdef |= !(fabs(P.rdiag[k]) >= 1e-12 * rmax);
    return rankdef;
}

// C = Q'HQ (reflector k from the left on every column, then from the right on every row); returns max|H|; every lane
TG_FN double tg_polish_reduce(const TgPolishWs &P, int nF, int nW)
{
    const int lane = TG_LANE();
    double hmax = 0;
    #pragma unroll 1
    for (size_t q = lane; q < (size_t)nF * nF; q += TG_NL) { P.C[q] = P.H[q]; hmax = tg_kkt_fold(hmax, fabs(P.H[q])); }
    int k0 = 0;
    tg_wargmax(hmax, k0);
    TG_SYNC();
    #pragma unroll 1
    for (int k = 0; k < nW; k++) {
        const double *v = P.AT + (size_t)k * nF, beta = P.beta[k];
        #pragma unroll 1
        for (int j = lane; j < nF; j += TG_NL) {
            double t = 0;
            #pragma unroll 1
            for (int a = k; a < nF; a++) t += v[a] * P.C[(size_t)a * nF + j];
            t *= beta;
            #pragma unroll 1
            for (int a = k; a < nF; a++) P.C[(size_t)a * nF + j] -= t * v[a];
        }
        TG_SYNC();
        #pragma unroll 1
        for (int i = lane; i < nF; i += TG_NL) {
            double *row = P.C + (size_t)i * nF;
            double t = 0;
            #pragma unroll 1
            for (int a = k; a < nF; a++) t += row[a] * v[a];
            t *= beta;
            #pragma unroll 1
            for (int a = k; a < nF; a++) row[a] -= t * v[a];
        }
        TG_SYNC();
    }
    return hmax;
}

// Cholesky of the reduced Hessian C[nW.., nW..] + delta I into F (lower triangle, row-major nz x nz, nz = nF - nW);
// returns 0 when a pivot is not positive and finite; every lane
TG_FN int tg_polish_chol(const TgPolishWs &P, int nF, int nW, double delta)
{
    const int lane = TG_LANE(), nz = nF - nW;
    #pragma unroll 1
    for (int q = lane; q < nz * nz; q += TG_NL) {
        const int a = q / nz, b = q - a * nz;
        P.F[q] = P.C[(size_t)(nW + a) * nF + nW + b] + (a == b ? delta : 0.0);
    }
    TG_SYNC();
    int ok = 1;
    #pragma unroll 1
    for (int k = 0; k < nz && ok; k++) {
        const double d = P.F[(size_t)k * nz + k];
        if (!(d > 0) || !tg_finite(d)) { ok = 0; break; }
        const double lkk = sqrt(d);
        TG_SYNC();
        if (lane == 0) P.F[(size_t)k * nz + k] = lkk;
        #pragma unroll 1
        for (int i = k + 1 + lane; i < nz; i += TG_NL) P.F[(size_t)i * nz + k] /= lkk;
        TG_SYNC();
        #pragma unroll 1
        for (int i = k + 1 + lane; i < nz; i += TG_NL) {
            const double lik = P.F[(size_t)i * nz + k];
            #pragma unroll 1
            for (int j = k + 1; j <= i; j++) P.F[(size_t)i * nz + j] -= lik * P.F[(size_t)j * nz + k];
        }
        TG_SYNC();
    }
    TG_SYNC();
    return ok;
}

// vec[0..nz) <- (F F')^-1 vec, forward then back substitution; one lane
TG_HD void tg_polish_chol_solve(const TgPolishWs &P, int nz, double *vec)
{
    for (int a = 0; a < nz; a++) {
        double s = vec[a];
        for (int b = 0; b < a; b++) s -= P.F[(size_t)a * nz + b] * vec[b];
        vec[a] = s / P.F[(size_t)a * nz + a];
    }
    for (int a = nz - 1; a >= 0; a--) {
        double s = vec[a];
        for (int b = a + 1; b < nz; b++) s -= P.F[(size_t)b * nz + a] * vec[b];
        vec[a] = s / P.F[(size_t)a * nz + a];
    }
}

// vec[0..nW) <- R^-1 vec, back substitution with the R of tg_polish_qr; one lane
TG_HD void tg_polish_rsolve(const TgPolishWs &P, int nF, int nW, double *vec)
{
    for (int k = nW - 1; k >= 0; k--) {
        double s = vec[k];
        for (int j = k + 1; j < nW; j++) s -= P.AT[(size_t)j * nF + k] * vec[j];
        vec[k] = s / P.rdiag[k];
    }
}

// Polishes one problem in place (see the top of the file).  sp / par: the problem's descriptor and parameter row;
// x[n], f, violation, lam[m], kkt[4]: its solve outputs, replaced only when the final guard holds.
template <int D>
TG_FN void tg_polish_problem(const TgLayout &L, const int *sp, const double *par, double *ws, double *xio, double *fio,
                             int status, int *violation, double *lamio, double *kktio, int *pstatus, int *piters,
                             int maxiter, double tol)
{
    const int lane = TG_LANE(), n = L.n, m = L.m, meq = L.meq;
    if (status != 0) {
        if (lane == 0) { *pstatus = TG_POLISH_SKIPPED; *piters = 0; }
        return;
    }
    TgPolishWs P;
    tg_polish_carve(L, ws, &P);
    #pragma unroll 1
    for (int i = lane; i < L.P; i += TG_NL) P.par[i] = par[i];
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) {
        tg_polish_bounds(L, i, P.xl[i], P.xu[i]);
        P.x[i] = P.xt[i] = xio[i];
    }
    double lmax = 0;
    #pragma unroll 1
    for (int j = lane; j < m; j += TG_NL) { P.lam[j] = lamio[j]; P.drop[j] = 0; lmax = tg_kkt_fold(lmax, fabs(lamio[j])); }
    #pragma unroll 1
    for (size_t q = lane; q < (size_t)m * n; q += TG_NL) P.J[q] = 0;
    int k0 = 0;
    tg_wargmax(lmax, k0);
    const double rho = 1 + 2 * lmax;
    TG_SYNC();
    {
        TgJac sink = {P.J, n, 1, 0};
        tg_linear_jacobian_d<D>(L, sp, P.par, sink);
    }
    double f = tg_polish_eval<D>(L, sp, P), gmax, kkt[4];
    tg_polish_kkt(L, P, P.lam, kkt, &gmax);
    const double v_in = tg_polish_maxviol(L, P.c), merit_in = tg_polish_merit(L, f, P.c, rho), st_in = kkt[0];
    double merit = merit_in;
    int it = 0, conv = 0, hvalid = 0, moved = 0;
    #pragma unroll 1
    for (;;) {
        if (kkt[0] <= tol * fmax(1.0, gmax)) { conv = 1; break; }
        if (it >= maxiter) break;
        // ---- free variables and working set
        int nF, nW;
        tg_polish_sets(L, P, &nF, &nW);
        if (nW > nF) {
            if (lane == 0) { *pstatus = TG_POLISH_DEGENERATE; *piters = it; }
            return;
        }
        // ---- Hessian of the Lagrangian over the free variables
        if (!hvalid) {
            tg_polish_hessian<D>(L, sp, P, nF);
            hvalid = 1;
        }
        // ---- Householder QR of A_W' (nF x nW, column k = row W_k over the free variables)
        if (tg_polish_qr(L, P, nF, nW)) {
            if (lane == 0) { *pstatus = TG_POLISH_DEGENERATE; *piters = it; }
            return;
        }
        // ---- C = Q'HQ, gq = Q'g_F
        const double hmax = tg_polish_reduce(P, nF, nW);
        if (lane == 0) {
            for (int a = 0; a < nF; a++) P.gq[a] = P.g[P.fr[a]];
            for (int k = 0; k < nW; k++) tg_polish_reflect(P, nF, k, P.gq);
            // range-space part: R' p_y = -c_W
            for (int k = 0; k < nW; k++) {
                double s = -P.c[P.wrow[k]];
                for (int j = 0; j < k; j++) s -= P.AT[(size_t)k * nF + j] * P.pq[j];
                P.pq[k] = s / P.rdiag[k];
            }
        }
        TG_SYNC();
        // ---- reduced Hessian C[nW.., nW..] + delta I, Cholesky into F
        const int nz = nF - nW;
        int chol_ok = nz == 0;
        #pragma unroll 1
        for (int attempt = 0; attempt < 4 && !chol_ok; attempt++)
            chol_ok = tg_polish_chol(P, nF, nW, attempt == 0 ? 0.0 : 1e-8 * hmax * (attempt == 1 ? 1.0 : attempt == 2 ? 1e2 : 1e4));
        if (!chol_ok) break;
        // null-space part: (Z'HZ) p_z = -(gq_z + C_zy p_y); rhs in tmp
        #pragma unroll 1
        for (int a = lane; a < nz; a += TG_NL) {
            const double *row = P.C + (size_t)(nW + a) * nF;
            double s = P.gq[nW + a];
            #pragma unroll 1
            for (int k = 0; k < nW; k++) s += row[k] * P.pq[k];
            P.tmp[a] = -s;
        }
        TG_SYNC();
        if (lane == 0) {
            tg_polish_chol_solve(P, nz, P.tmp);
            for (int a = 0; a < nz; a++) P.pq[nW + a] = P.tmp[a];
        }
        TG_SYNC();
        // ---- multipliers: R lam_W = gq_y + (C pq)_y
        #pragma unroll 1
        for (int k = lane; k < nW; k += TG_NL) {
            const double *row = P.C + (size_t)k * nF;
            double s = P.gq[k];
            #pragma unroll 1
            for (int b = 0; b < nF; b++) s += row[b] * P.pq[b];
            P.tmp[k] = s;
        }
        TG_SYNC();
        if (lane == 0) {
            tg_polish_rsolve(P, nF, nW, P.tmp);
            for (int j = 0; j < m; j++) P.lamw[j] = 0;
            for (int k = 0; k < nW; k++) P.lamw[P.wrow[k]] = P.tmp[k];
            // step over the free variables: p_F = Q pq
            for (int k = nW - 1; k >= 0; k--) tg_polish_reflect(P, nF, k, P.pq);
        }
        TG_SYNC();
        // ---- an inequality row with a negative multiplier leaves W (the most negative one; ties: the first row)
        int jneg = -1;
        double lneg = 0;
        #pragma unroll 1
        for (int k = 0; k < nW; k++) {
            const int j = P.wrow[k];
            if (j >= meq && P.lamw[j] < lneg) { lneg = P.lamw[j]; jneg = j; }
        }
        if (jneg >= 0) {
            TG_SYNC();
            if (lane == 0) P.drop[jneg] = 1;
            TG_SYNC();
            it++;
            continue;
        }
        // ---- backtracking on the merit; the trial x clipped to the bounds
        int accepted = 0;
        #pragma unroll 1
        for (int t = 0; t < 4 && !accepted; t++) {
            const double step = t == 0 ? 1.0 : t == 1 ? 0.5 : t == 2 ? 0.25 : 0.125;
            #pragma unroll 1
            for (int a = lane; a < nF; a += TG_NL) {
                const int i = P.fr[a];
                P.xt[i] = fmin(fmax(P.x[i] + step * P.pq[a], P.xl[i]), P.xu[i]);
            }
            TG_SYNC();
            const double ft = tg_objective(L, sp, P.xt, 0);
            tg_constraints_d<D>(L, sp, P.par, P.xt, P.ct, 0, P.scratch);
            TG_SYNC();
            const double mt = tg_polish_merit(L, ft, P.ct, rho);
            accepted = mt <= merit;
        }
        it++;
        if (!accepted) {
            #pragma unroll 1
            for (int i = lane; i < n; i += TG_NL) P.xt[i] = P.x[i];
            TG_SYNC();
            break;
        }
        #pragma unroll 1
        for (int i = lane; i < n; i += TG_NL) P.x[i] = P.xt[i];
        #pragma unroll 1
        for (int j = lane; j < m; j += TG_NL) { P.lam[j] = P.lamw[j]; P.drop[j] = 0; }
        TG_SYNC();
        moved = 1; hvalid = 0;
        f = tg_polish_eval<D>(L, sp, P);
        tg_polish_kkt(L, P, P.lam, kkt, &gmax);
        merit = tg_polish_merit(L, f, P.c, rho);
    }
    // ---- final guard
    bool finite = tg_finite(f);
    double lm = 0;
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) finite = finite && tg_finite(P.x[i]);
    #pragma unroll 1
    for (int j = lane; j < m; j += TG_NL) { finite = finite && tg_finite(P.lam[j]); lm = tg_kkt_fold(lm, fabs(P.lam[j])); }
    for (int q = 0; q < 4; q++) finite = finite && tg_finite(kkt[q]);
    finite = !tg_any(!finite);
    tg_wargmax(lm, k0);
    const double v_out = tg_polish_maxviol(L, P.c);
    const bool keep = moved && finite && v_out <= fmax(v_in, 1e-8) && merit <= merit_in && kkt[0] < st_in &&
                      kkt[2] <= 1e-8 * fmax(1.0, lm);
    if (!keep) {
        if (lane == 0) { *pstatus = moved && !finite ? TG_POLISH_NONFINITE : TG_POLISH_REJECTED; *piters = it; }
        return;
    }
    const int viol = tg_last_block_violation(L, P.c);
    #pragma unroll 1
    for (int i = lane; i < n; i += TG_NL) xio[i] = P.x[i];
    #pragma unroll 1
    for (int j = lane; j < m; j += TG_NL) lamio[j] = P.lam[j];
    if (lane == 0) {
        *fio = f; *violation = viol;
        for (int q = 0; q < 4; q++) kktio[q] = kkt[q];
        *pstatus = conv ? TG_POLISH_POLISHED : TG_POLISH_IMPROVED; *piters = it;
    }
    TG_SYNC();
}

#endif  // TG_POLISH_H
