// TEST INFRASTRUCTURE -- the host build with the certificate (tg_hostsim_kkt.cpp) plus the post-solve polish
// (csrc/tg_polish.h), for tests/test_polish.py.  Never loaded by the product.
#include "tg_hostsim_kkt.cpp"
#include "../../trajectory_generator_b200/csrc/tg_polish.h"

// tg_polish_problem on one problem: x[n], f, violation, lam[m], kkt[4] updated in place
extern "C" void hs_polish(const int *spec, const double *par, double *x, double *f, int status, int *violation, double *lam,
                          double *kkt, int *pstatus, int *piters, int maxiter, double tol)
{
    TgLayout L;
    tg_make_layout(spec, &L);
    std::vector<double> ws(tg_polish_group_doubles(L));
    if (L.d == 2) tg_polish_problem<2>(L, spec, par, ws.data(), x, f, status, violation, lam, kkt, pstatus, piters, maxiter, tol);
    else tg_polish_problem<3>(L, spec, par, ws.data(), x, f, status, violation, lam, kkt, pstatus, piters, maxiter, tol);
}
