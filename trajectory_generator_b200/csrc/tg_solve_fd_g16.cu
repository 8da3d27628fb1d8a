// M2 stage FD (finite-difference mode), 16 lanes per problem: the forward-difference sweeps as a kernel of their own,
// with the evaluators inlined value-only (see tg_kernels_solve.inc)
#define TG_GS 16
#define TG_INLINE_ALL
#define TG_DER_STAGE
#define TG_SFX _g16
// fixed shapes (tg_shape.h) with instantiations in this translation unit: the BASELINE configurations this group size serves
#define TG_LS_FIXED TG_FIXED_CASE(TG_FIX_C3) TG_FIXED_CASE(TG_FIX_C4)
#include "tg_kernels_solve.inc"
