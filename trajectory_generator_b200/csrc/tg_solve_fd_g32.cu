// M2 stage FD (finite-difference mode), 32 lanes per problem: the forward-difference sweeps as a kernel of their own,
// with the evaluators inlined value-only (see tg_kernels_solve.inc)
#define TG_GS 32
#define TG_INLINE_ALL
#define TG_DER_STAGE
#define TG_SFX _g32
#include "tg_kernels_solve.inc"
