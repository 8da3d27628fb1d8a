// TEST INFRASTRUCTURE -- the single-lane host build (tg_hostsim.cpp) plus the multipliers and the KKT certificate of a
// finished solve (csrc/tg_sqp.h, tg_sqp_kkt), for tests/test_multipliers.py.  Never loaded by the product.
#include "tg_hostsim.cpp"

#ifdef TG_WITH_SQP
// hs_solve plus the multipliers lam[m] and the KKT certificate kkt[4] of the final state
extern "C" int hs_solve_kkt(const int *spec, const double *par, double *x, int maxiter, double ftol, int flags, double *fout,
                            int *status, int *nit, int *nfev, double *lam, double *kkt)
{
    TgLayout L;
    tg_make_layout(spec, &L);
    std::vector<double> ws(tg_sqp_workspace_doubles(L)), scratch(tg_sqp_kkt_scratch_doubles(L) + 1);
    TgSqpResult res;
    if (L.d == 2) tg_sqp_solve<2>(L, spec, par, x, ws.data(), maxiter, ftol, flags, &res, nullptr, 0);
    else tg_sqp_solve<3>(L, spec, par, x, ws.data(), maxiter, ftol, flags, &res, nullptr, 0);
    TgSqpWs W;
    tg_sqp_carve(L, ws.data(), &W);
    tg_sqp_kkt(L, W, lam, kkt, scratch.data());
    *fout = res.f; *status = res.status; *nit = res.nit; *nfev = res.nfev;
    return res.status;
}
#endif
