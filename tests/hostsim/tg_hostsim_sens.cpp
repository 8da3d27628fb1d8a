// TEST INFRASTRUCTURE -- the host build with the certificate and the polish (tg_hostsim_polish.cpp) plus the parameter
// sensitivities (csrc/tg_sens.h), for tests/test_sensitivity.py.  Never loaded by the product.
#include "tg_hostsim_polish.cpp"
#include "../../trajectory_generator_b200/csrc/tg_sens.h"

// tg_sens_problem on one problem: par_bar[P] and the status code
extern "C" void hs_sens(const int *spec, const double *par, const double *x, int status, const double *lam,
                        const double *xbar, double fbar, double *pbar, int *sstatus, double tol)
{
    TgLayout L;
    tg_make_layout(spec, &L);
    std::vector<double> ws(tg_sens_group_doubles(L));
    if (L.d == 2) tg_sens_problem<2>(L, spec, par, ws.data(), x, status, lam, xbar, fbar, pbar, sstatus, tol);
    else tg_sens_problem<3>(L, spec, par, ws.data(), x, status, lam, xbar, fbar, pbar, sstatus, tol);
}
